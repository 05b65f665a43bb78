"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Bar: bit-exact -- identical site lists (motif, sequence, start, strand, in order) and identical
doubles for every score.  No tolerance anywhere in this file.
"""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

KAT_M = [[[1.35, 0.21, -5.23], [0.07, -0.21, 0.6], [2.15, 2.22, -0.84], [-2.64, -1.89, 5.47]]]


@pytest.fixture(scope="module")
def cs():
    from motifscan_b200.motif import cscore
    return cscore


@pytest.fixture(scope="module")
def eng():
    from motifscan_b200 import engine
    return engine


def synth_pwms(rng, n, lmin=6, lmax=30, bg=(0.295, 0.205, 0.205, 0.295)):
    """Production-shaped PWMs: PFM -> PPM (pseudo 0.001) -> log-odds rounded to 5 dp."""
    out = []
    for _ in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        depth = int(np.exp(rng.uniform(np.log(20), np.log(5000))))
        pfm = np.round(depth * rng.dirichlet([0.3] * 4, size=L).T).astype(np.int64)
        pfm[0, pfm.sum(axis=0) == 0] = 1
        out.append(oracle.pfm_to_pwm(pfm, dict(zip("ACGT", bg))).tolist())
    return out


def synth_seqs(rng, n, lo, hi, p_n=0.0, p_lower=0.3, n_blocks=False):
    alphabet = np.frombuffer(b"ACGT", dtype=np.uint8)
    out = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        s = alphabet[rng.choice(4, size=L, p=[0.295, 0.205, 0.205, 0.295])].copy()
        low = rng.random(L) < p_lower
        s[low] |= 0x20
        if p_n > 0:
            s[rng.random(L) < p_n] = ord("N")
        if n_blocks and L > 200:
            a = int(rng.integers(0, L - 100))
            s[a:a + int(rng.integers(1, 100))] = ord("N")
            s[:int(rng.integers(0, 40))] = ord("n")
        out.append(bytes(s).decode())
    return out


def cutoffs_for(pwms, seqs, rate):
    """Score cutoffs putting roughly `rate` of the windows above the cutoff (from the oracle's
    offset-0 scores of random sub-windows; only a way to pick realistic thresholds)."""
    rng = np.random.default_rng(1)
    lmax = max(len(p[0]) for p in pwms)
    pool = [s for s in seqs if len(s) >= lmax + 1]
    samples = []
    for _ in range(4000):
        s = pool[int(rng.integers(len(pool)))]
        a = int(rng.integers(0, len(s) - lmax + 1))
        samples.append(s[a:a + lmax].upper().replace("N", "A"))
    sc = oracle.score_arrays(pwms, samples, 3)
    k = max(int(len(samples) * rate), 1)
    return [float(np.sort(row)[::-1][k]) for row in sc]


def assert_scan_equal(res, expect):
    counts, seq_idx, start, score, strand = expect
    assert np.array_equal(res.counts, counts)
    assert np.array_equal(res.seq_idx, seq_idx.astype(np.int32))
    assert np.array_equal(res.start, start.astype(np.int32))
    assert np.array_equal(res.strand, strand)
    # bit-exact doubles (also distinguishes -0.0 / 0.0 and NaN payloads)
    assert np.array_equal(res.score.view(np.uint64), score.view(np.uint64))


def test_kat_c_score(cs):
    # reference tests/test_motif_score.py:6-20
    seqs = ['NNN', 'AGT', 'ANT', 'CTA']
    assert cs.c_score(KAT_M, seqs, 1, 1)[0] == pytest.approx(
        [0.0, 0.9186991869918698, 0.693089430894309, -0.7164634146341464])
    assert cs.c_score(KAT_M, seqs, 2, 1)[0] == pytest.approx(
        [0.0, 0.6717479674796748, 0.693089430894309, -0.3323170731707317])
    assert cs.c_score(KAT_M, seqs, 3, 1)[0] == pytest.approx(
        [0.0, 0.9186991869918698, 0.693089430894309, -0.3323170731707317])


def test_kat_c_scan_motif(cs):
    # reference tests/test_motif_score.py:23-32
    motif_sites = cs.c_scan_motif(KAT_M, [0.2], ['NNNAG', 'TANTCTA'], 3, 1)
    assert len(motif_sites) == 1
    assert len(motif_sites[0]) == 4
    assert motif_sites[0][0] == pytest.approx([1, 1, 0.693089430894309, 1])
    assert motif_sites[0][1] == pytest.approx([1, 1, 0.693089430894309, 2])
    assert motif_sites[0][2] == pytest.approx([1, 2, 0.23983739837398374, 2])
    assert motif_sites[0][3] == pytest.approx([1, 3, 0.266260162601626, 1])


def test_golden_cases_bit_exact(cs, cscore_cases):
    """Fixtures produced by the unmodified reference extension (tests/golden/make_golden.py)."""
    for c in cscore_cases:
        got = cs.c_scan_motif(c["pwms"], c["cutoffs"], c["seqs"], c["strand"], 1)
        assert got == c["scan"], c["name"]
        if c["score_seqs"]:
            assert cs.c_score(c["pwms"], c["score_seqs"], c["strand"], 1) == c["score"], c["name"]


def test_encoding_bit_exact(eng):
    """2-bit + mask packing decodes to exactly the reference's int8 codes (cscore.c:81-114)."""
    rng = np.random.default_rng(3)
    every_byte = bytes(range(1, 128)).decode("ascii")
    seqs = [every_byte, "", "A", "acgtn" * 13, "N" * 70] + synth_seqs(rng, 40, 0, 700, p_n=0.05, n_blocks=True)
    seqs.append("ACGTé中acgt")  # multi-byte UTF-8: every byte of it is "N" (cscore.c:83)
    ctx = eng.default_context(0)
    sset = eng.SequenceSet(ctx, seqs)
    blob = "".join(seqs).encode("utf-8")
    assert np.array_equal(sset.codes(), oracle.encode(blob))
    sset.close()


@pytest.mark.parametrize("strand", [1, 2, 3])
def test_random_production_shape(eng, strand):
    rng = np.random.default_rng(100 + strand)
    pwms = synth_pwms(rng, 60)
    seqs = synth_seqs(rng, 300, 900, 1100)
    cutoffs = cutoffs_for(pwms, seqs, 2e-3)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, strand)
    assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8))
    assert res.n_sites > 100
    res.close(), sset.close(), motifs.close()


def test_n_blocks_lowercase_and_ragged(eng):
    rng = np.random.default_rng(7)
    pwms = synth_pwms(rng, 40, lmin=1, lmax=32)
    seqs = synth_seqs(rng, 120, 0, 1500, p_n=0.01, n_blocks=True)
    seqs += ["", "A", "N", "ACGTACGTAC", "n" * 100, "NNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNACGTACGTTTGACCA"]
    cutoffs = cutoffs_for(pwms, seqs, 5e-3)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    for strand in (3, 1, 2):
        res = eng.scan(ctx, motifs, sset, strand)
        assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8))
        res.close()
    sset.close(), motifs.close()


def test_zero_score_windows_hit_when_cutoff_allows(eng):
    """All-N windows score exactly 0 and are sites when cutoff <= 1e-10 (cscore.c:358)."""
    rng = np.random.default_rng(8)
    pwms = synth_pwms(rng, 5, lmin=4, lmax=12)
    seqs = ["N" * 80, "ACGT" * 10 + "N" * 50 + "ACGT" * 10, "n" * 33]
    cutoffs = [0.0, 1e-10, 1e-9, -0.5, 0.7]
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, 3)
    assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, 3))
    assert res.counts[0] > 100
    res.close(), sset.close(), motifs.close()


def test_many_motifs_multiple_batches(eng):
    """More motifs than fit one shared-memory batch (> 24 tensor-core tile steps / > 227 KB of tables)."""
    rng = np.random.default_rng(11)
    pwms = synth_pwms(rng, 2100, lmin=6, lmax=30)
    seqs = synth_seqs(rng, 24, 400, 600)
    cutoffs = cutoffs_for(pwms, seqs, 1e-3)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, 3)
    assert ctx.counters()["prefilter_launches"] >= 2
    assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, 3, n_threads=8))
    res.close(), sset.close(), motifs.close()


def test_arbitrary_float_int_and_degenerate_pwms(eng):
    rng = np.random.default_rng(12)
    pwms = [rng.normal(0, 2, size=(4, int(rng.integers(1, 33)))).tolist() for _ in range(20)]
    pwms += [rng.integers(-3, 4, size=(4, int(rng.integers(2, 10)))).astype(float).tolist() for _ in range(10)]
    pwms.append((-np.abs(rng.normal(0, 1, size=(4, 7))) - 0.1).tolist())  # max_raw == 0: never a site
    pwms.append(np.zeros((4, 5)).tolist())                                   # 0/0 = NaN: never a site
    pwms.append(np.full((4, 6), 2.5).tolist())                               # constant: every window 1.0
    pwms.append(rng.normal(0, 2, size=(4, 45)).tolist())                     # L > 32: exact path
    pwms.append(rng.normal(0, 2, size=(4, 33)).tolist())
    seqs = synth_seqs(rng, 30, 0, 400, p_n=0.02, n_blocks=True)
    cutoffs = [float(rng.uniform(0.1, 0.7)) for _ in pwms]
    cutoffs[3] = float("nan")
    cutoffs[4] = float("inf")
    cutoffs[5] = float("-inf")
    cutoffs[6] = -2.0   # everything is a site
    cutoffs[7] = 5.0    # nothing is
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    for strand in (3, 1, 2):
        res = eng.scan(ctx, motifs, sset, strand)
        assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8))
        res.close()
    sset.close(), motifs.close()


def test_long_motifs_production_shape(eng):
    """Motifs longer than 32 columns: the tensor-core prefilter looks at the first 32 columns of each strand
    and the exact stage scores the whole window from memory (N anywhere in it, also behind base 32); motifs
    longer than 64 columns take the every-position exact kernel.  The oracle's sites, bit for bit."""
    rng = np.random.default_rng(121)
    pwms = synth_pwms(rng, 24, lmin=33, lmax=64) + synth_pwms(rng, 40, lmin=6, lmax=32) + synth_pwms(rng, 2, lmin=65, lmax=80)
    seqs = synth_seqs(rng, 80, 200, 1500, p_n=0.004, n_blocks=True) + ["ACGT" * 8 + "A", "N" * 70, "acgt" * 16 + "N" + "acgt" * 9]
    # runs of N followed by sequence: a window whose first 32 bases are N still scores > 0 for a longer motif
    seqs += ["N" * 100 + s[:120] + "N" * 40 + s[120:300] for s in synth_seqs(rng, 12, 300, 300)]
    cutoffs = cutoffs_for(pwms, seqs, 3e-3)
    for m in (0, 3, 7, 30):
        cutoffs[m] = 1e-6          # nearly every window with a positive partial score is a site (incl. mostly-N ones)
    ctx = eng.Context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    for strand in (3, 1, 2):
        expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
        res = eng.scan(ctx, motifs, sset, strand)
        assert_scan_equal(res, expect)
        assert int(expect[0][:24].sum()) > 200          # the long motifs do have sites
        res.close()
    sset.close(), motifs.close(), ctx.close()


def test_dense_hits_overflow_retry(eng):
    """Cutoffs so low that candidates overflow the first buffers: results must not change."""
    rng = np.random.default_rng(13)
    pwms = synth_pwms(rng, 30, lmin=6, lmax=12)
    seqs = synth_seqs(rng, 100, 1900, 2100)
    cutoffs = [-5.0] * len(pwms)
    ctx = eng.Context(0)  # fresh context: scratch starts at its minimum size
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, 3)
    assert ctx.counters()["retries"] >= 1
    assert_scan_equal(res, oracle.scan_arrays(pwms, cutoffs, seqs, 3, n_threads=8))
    res.close(), sset.close(), motifs.close(), ctx.close()


def test_lane_record_buffer_overflow_retry(eng):
    """Tensor-core prefilter: every epilogue lane appends candidate records to its own buffer; a lane
    that runs out of room only counts, and the scan is repeated with buffers sized for the largest
    count.  Forced here with a first-attempt capacity of 2 records per lane."""
    from motifscan_b200 import _lib
    rng = np.random.default_rng(113)
    pwms = synth_pwms(rng, 200)
    seqs = synth_seqs(rng, 40, 900, 1100, p_n=0.001)
    cutoffs = cutoffs_for(pwms, seqs, 2e-3)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    expect = oracle.scan_arrays(pwms, cutoffs, seqs, 3, n_threads=8)
    try:
        ctx.set_option("tc_first_lane_cap", 2)
        res = eng.scan(ctx, motifs, sset, 3)
        assert ctx.counters()["retries"] >= 1
        assert_scan_equal(res, expect)
        res.close()
    finally:
        ctx.set_option("tc_first_lane_cap", 0)
    res = eng.scan(ctx, motifs, sset, 3)
    assert ctx.counters()["retries"] == 0
    assert_scan_equal(res, expect)
    res.close(), sset.close(), motifs.close()


def test_set_cutoffs_rebuilds_tables(eng):
    rng = np.random.default_rng(14)
    pwms = synth_pwms(rng, 12)
    seqs = synth_seqs(rng, 50, 500, 600)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, [0.9] * 12)
    sset = eng.SequenceSet(ctx, seqs)
    for cut in (0.9, 0.6, 0.75):
        motifs.set_cutoffs([cut] * 12)
        res = eng.scan(ctx, motifs, sset, 3)
        assert_scan_equal(res, oracle.scan_arrays(pwms, [cut] * 12, seqs, 3, n_threads=8))
        res.close()
    sset.close(), motifs.close()


@pytest.mark.parametrize("strand", [1, 2, 3])
def test_tensor_prefilter_sites_and_candidate_density(eng, strand):
    """The tensor-core prefilter is conservative: after the exact stage it gives the oracle's sites.  It
    does not flood the exact stage with candidates either.  The option that selected the former
    shared-memory table prefilter is refused, not ignored."""
    rng = np.random.default_rng(150 + strand)
    pwms = synth_pwms(rng, 300)
    seqs = synth_seqs(rng, 150, 700, 1300, p_n=0.002, n_blocks=True)
    cutoffs = cutoffs_for(pwms, seqs, 5e-4)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
    with pytest.raises(ValueError):
        ctx.set_option("prefilter_tc", 0)
    res = eng.scan(ctx, motifs, sset, strand)
    assert_scan_equal(res, expect)
    # No flood: at most 2.9 candidate records per oracle site in a window of A/C/G/T only.  Only those windows
    # go through the prefilter: here 97 % of the sites touch an N (negative cutoffs, N adds 0) and are scored by
    # the dirty-window kernel.  2.9 is the largest one-decimal k with k * clean sites <= 3 * (candidates of the
    # former table prefilter) on every strand of these inputs, measured on a B200, so the bound is no looser
    # than the former one of 3x the table prefilter's candidates.
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    not_acgt = np.concatenate([[0], np.cumsum(~np.isin(blob, np.frombuffer(b"ACGTacgt", dtype=np.uint8)))])
    first = np.concatenate([[0], np.cumsum([len(s) for s in seqs])])[expect[1]] + expect[2]
    last = first + np.repeat([len(p[0]) for p in pwms], expect[0])
    clean_sites = int(np.count_nonzero(not_acgt[last] == not_acgt[first]))
    cand = ctx.counters()["candidates"]
    assert cand <= 2.9 * clean_sites + 1000, (cand, clean_sites)
    res.close(), sset.close(), motifs.close()


def test_score_matches_oracle_bit_exact(eng):
    rng = np.random.default_rng(16)
    pwms = synth_pwms(rng, 70, lmin=1, lmax=30)
    pwms.append(rng.normal(0, 2, size=(4, 40)).tolist())
    seqs = synth_seqs(rng, 3000, 40, 60, p_n=0.01)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms)
    sset = eng.SequenceSet(ctx, seqs)
    for strand in (1, 2, 3):
        got = eng.score(ctx, motifs, sset, strand)
        want = oracle.score_arrays(pwms, seqs, strand)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    with pytest.raises(ValueError):
        short = eng.SequenceSet(ctx, ["ACGTACGT"])
        eng.score(ctx, motifs, short, 3)
    sset.close(), motifs.close()


def test_score_select_matches_sorted_order_statistics(eng):
    """Fused score + order statistics == sorting the oracle's scores (motif/__init__.py:396-399)."""
    rng = np.random.default_rng(17)
    pwms = synth_pwms(rng, 25)
    seqs = synth_seqs(rng, 20000, 30, 30)
    n = len(seqs)
    ranks = [int(n * 0.1 ** e) - 1 for e in range(2, min(len(str(n)), 7))]
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms)
    sset = eng.SequenceSet(ctx, seqs)
    got = eng.score_select(ctx, motifs, sset, 3, ranks)
    want = oracle.score_arrays(pwms, seqs, 3)
    want = np.sort(want, axis=1)[:, ::-1][:, ranks]
    assert np.array_equal(got.view(np.uint64), np.ascontiguousarray(want).view(np.uint64))
    sset.close(), motifs.close()


@pytest.mark.parametrize("nudge", ["exact", "plus_1e-10", "next_double_up", "minus_half_quantum"])
def test_cutoffs_placed_on_window_scores_lose_no_site(eng, nudge):
    """The tensor-core prefilter must flag a SUPERSET of the reference's hits although it works with e4m3 entries
    and f16 accumulators (one rounding per K step, prefilter_tc.cuh).  Adversarial placement: every motif's
    cutoff sits exactly on the score of real windows of the input (so whole groups of windows are borderline:
    score - cutoff = 0, or -1e-10 exactly, or one ulp short), or half an e4m3 quantum below them.  A window the
    prefilter dropped could not come back, so equality with the oracle at site level is the superset property
    at candidate level; the candidate counter is checked to be at least the number of sites as well."""
    rng = np.random.default_rng(190)
    pwms = synth_pwms(rng, 120, lmin=4, lmax=32)
    seqs = synth_seqs(rng, 60, 500, 900, p_n=0.002, n_blocks=True)
    loose = cutoffs_for(pwms, seqs, 5e-3)
    counts, _, _, score, _ = oracle.scan_arrays(pwms, loose, seqs, 3, n_threads=8)
    off = np.concatenate([[0], np.cumsum(counts)])
    cutoffs = []
    for m, p in enumerate(pwms):
        sc = np.sort(score[off[m]:off[m + 1]])
        if len(sc) == 0:
            cutoffs.append(loose[m])
            continue
        c = float(sc[len(sc) // 2])                       # the score of actual windows of this input
        if nudge == "plus_1e-10":
            c = c + 1e-10
        elif nudge == "next_double_up":
            c = float(np.nextafter(c, np.inf))
        elif nudge == "minus_half_quantum":
            # one e4m3 step of the prefilter entries is ~1/16 of an entry; in score units that is about
            # (sum colmax - T) / (C * 16) / max_raw with C = L * beta ~ 384
            mat = np.asarray(p)
            c = c - 0.5 * float(np.abs(mat).max(axis=0).sum()) / (384 * 16) / max(oracle.max_raw_score(p), 1e-9)
        cutoffs.append(c)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    for strand in (3, 1, 2):
        expect = oracle.scan_arrays(pwms, cutoffs, seqs, strand, n_threads=8)
        res = eng.scan(ctx, motifs, sset, strand)
        assert_scan_equal(res, expect)
        c = ctx.counters()
        assert c["hits"] == int(expect[0].sum()) > 2000
        # a candidate record covers a (window, 64-column chunk): every site needs a flagged column in one
        assert c["candidates"] + c["dirty"] * len(pwms) * 2 >= np.count_nonzero(expect[0])
        res.close()
    sset.close(), motifs.close()


def test_long_sequence_dedup_equals_reference_rule(eng):
    """Device de-duplication walks chains of overlapping sites, not whole (motif, sequence) segments: on a few
    long sequences (many sites per segment, runs of N whose all-zero windows tie) it must keep exactly the sites
    the reference's pass keeps (scanner.py:156-193)."""
    rng = np.random.default_rng(191)
    pwms = synth_pwms(rng, 30, lmin=4, lmax=20)
    seqs = synth_seqs(rng, 3, 60000, 90000, p_n=0.0005, n_blocks=True)
    seqs[1] = seqs[1][:20000] + "N" * 3000 + seqs[1][23000:]
    cutoffs = cutoffs_for(pwms, seqs, 2e-2)
    cutoffs[0] = 0.0          # every all-N window of motif 0 is a site with score 0: one long chain of ties
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, 3, remove_dup=True)
    raw = oracle.c_scan_motif(pwms, cutoffs, seqs, 3, 8)
    want = oracle.deduplicate_motif_sites(oracle.make_motif_sites(raw, [0] * len(seqs)), [len(p[0]) for p in pwms])
    flat = [(m, r, s.start, s.score, 1 if s.strand == "+" else 2) for m, per in enumerate(want) for r, cell in enumerate(per) for s in cell]
    assert res.n_sites == len(flat) > 5000 and res.n_sites < sum(len(x) for x in raw)
    assert np.array_equal(res.seq_idx, np.array([f[1] for f in flat], dtype=np.int32))
    assert np.array_equal(res.start, np.array([f[2] for f in flat], dtype=np.int32))
    assert np.array_equal(res.strand, np.array([f[4] for f in flat], dtype=np.int8))
    assert np.array_equal(res.score.view(np.uint64), np.array([f[3] for f in flat]).view(np.uint64))
    res.close(), sset.close(), motifs.close()


def test_score_select_pilot_path_equals_sorting_every_score(eng):
    """msb_score_select on a large sample takes the pilot + scan + radix-select path (no score matrix): the
    order statistics must be the bits a full descending sort of the oracle's scores gives, for ordinary
    motifs, for motifs with a handful of distinct scores (heavy ties at every rank), for a motif whose scores
    are all NaN (0 / 0) and one whose windows all score the same, on every strand; and the same as the plain
    form (select_pilot = 0)."""
    from motifscan_b200 import _lib, synth
    rng = np.random.default_rng(170)
    pwms = synth_pwms(rng, 10) + synth_pwms(rng, 3, lmin=2, lmax=3)
    pwms.append([[0.0] * 5] * 4)                                   # max_raw = 0: every score is 0 / 0 = NaN
    pwms.append([[0.25] * 7] * 4)                                  # every window scores exactly 1
    pwms.append(np.around(rng.normal(0, 1, size=(4, 30)), 5).tolist())
    n = 300000
    blob, off = synth.background_samples(n, 30, seed=5)
    blob = blob.copy()
    blob[30 * 7 + 3] = ord("N")                                    # a sample with a non-ACGT base
    raw = blob.tobytes()
    seqs = [raw[off[i]:off[i + 1]].decode() for i in range(n)]
    ranks = [int(n * 0.1 ** e) - 1 for e in range(2, min(len(str(n)), 7))] + [0]
    ctx = eng.Context(0)
    motifs = eng.MotifSet(ctx, pwms)
    sset = eng.SequenceSet(ctx, blob=blob, seq_off=off)
    for strand in (3, 1, 2):
        want = np.sort(oracle.score_arrays(pwms, seqs, strand), axis=1)[:, ::-1][:, ranks]
        got = eng.score_select(ctx, motifs, sset, strand, ranks)
        redone = ctx.counters()["retries"]
        ctx.set_option("select_pilot", 0)
        plain = eng.score_select(ctx, motifs, sset, strand, ranks)
        ctx.set_option("select_pilot", 1)
        finite = ~np.isnan(want).any(axis=1)
        assert finite.sum() == len(pwms) - 1
        assert np.array_equal(got[finite].view(np.uint64), np.ascontiguousarray(want[finite]).view(np.uint64)), strand
        assert np.array_equal(got.view(np.uint64), plain.view(np.uint64))      # NaN rows: the same bits either way
        assert np.isnan(got[~finite]).all()
        assert 1 <= redone <= 3, redone                                         # the NaN motif (and nothing ordinary) is redone
    sset.close(), motifs.close(), ctx.close()


def test_scan_ascii_sliced_upload_equals_two_step_scan(eng):
    """msb_scan_ascii (upload cut into slices that overlap the scan; >= 8 MB takes the sliced path)
    == msb_seqs_from_ascii + msb_scan, from pinned and from pageable memory, with and without
    de-duplication; ragged sequences so that slice boundaries fall at odd packed positions."""
    rng = np.random.default_rng(77)
    pwms = synth_pwms(rng, 24)
    seqs = synth_seqs(rng, 6000, 900, 2100, p_n=0.0005, n_blocks=True)
    seqs += ["", "ACGT", "N" * 50]
    cutoffs = cutoffs_for(pwms, seqs, 2e-4)
    from motifscan_b200 import _lib
    blob, off = _lib.flatten_seqs(seqs)
    assert blob.size >= (8 << 20)
    ctx = eng.default_context(0)
    motifs = eng.MotifSet(ctx, pwms, cutoffs)
    sset = eng.SequenceSet(ctx, blob=blob, seq_off=off)
    pinned = eng.PinnedArray(blob.size)
    pinned.array[:] = blob
    for dedup in (False, True):
        want = eng.scan(ctx, motifs, sset, 3, remove_dup=dedup)
        for src in (pinned.array, blob):
            got = eng.scan_ascii(ctx, motifs, src, off, 3, remove_dup=dedup)
            assert got.n_sites == want.n_sites > 1000
            assert np.array_equal(got.counts, want.counts) and np.array_equal(got.seq_idx, want.seq_idx)
            assert np.array_equal(got.start, want.start) and np.array_equal(got.strand, want.strand)
            assert np.array_equal(got.score.view(np.uint64), want.score.view(np.uint64))
            got.close()
        want.close()
    small = eng.scan_ascii(ctx, motifs, blob[:off[40]], off[:41], 3)     # below the slicing threshold
    ref = oracle.scan_arrays(pwms, cutoffs, seqs[:40], 3, n_threads=4)
    assert_scan_equal(small, ref)
    small.close(), pinned.close(), sset.close(), motifs.close()


def test_sliced_scan_after_a_differently_sized_scan_with_a_poisoned_pool(eng):
    """The device buffers of a sequence set come from a recycling pool.  msb_scan_ascii scans slice k
    before slice k + 1 is encoded, and the last position tile of a slice reaches into the next slice's
    blocks: nothing there (codes, mask, block-owner table) may be read as if it were valid.  The pool
    is poisoned (0xFF) between two sliced scans of different shapes; results must still be the
    two-step scan's, which is checked against the oracle on a prefix."""
    from motifscan_b200 import _lib
    rng = np.random.default_rng(177)
    pwms = synth_pwms(rng, 16)
    ctx = eng.Context(0)
    ctx.set_option("poison_pool", 1)
    try:
        for n, lo, hi in ((5000, 1500, 2500), (9000, 800, 1200), (2500, 3300, 3500)):
            seqs = synth_seqs(rng, n, lo, hi, p_n=0.0005, n_blocks=True)
            cutoffs = cutoffs_for(pwms, seqs[:200], 5e-4)
            blob, off = _lib.flatten_seqs(seqs)
            assert blob.size >= (8 << 20)
            motifs = eng.MotifSet(ctx, pwms, cutoffs)
            got = eng.scan_ascii(ctx, motifs, blob, off, 3)
            sset = eng.SequenceSet(ctx, blob=blob, seq_off=off)
            want = eng.scan(ctx, motifs, sset, 3)
            assert got.n_sites == want.n_sites > 1000
            assert np.array_equal(got.counts, want.counts) and np.array_equal(got.seq_idx, want.seq_idx)
            assert np.array_equal(got.start, want.start) and np.array_equal(got.strand, want.strand)
            assert np.array_equal(got.score.view(np.uint64), want.score.view(np.uint64))
            head = eng.scan_ascii(ctx, motifs, blob[:off[300]], off[:301], 3)
            assert_scan_equal(head, oracle.scan_arrays(pwms, cutoffs, seqs[:300], 3, n_threads=8))
            head.close(), got.close(), want.close(), sset.close(), motifs.close()
    finally:
        ctx.close()


def test_threads_sharing_a_context_are_serialised(eng):
    """Two host threads scanning on the same context (what two Scanners on the default context do):
    the engine serialises the calls, results are the oracle's."""
    import threading
    rng = np.random.default_rng(91)
    pwms = synth_pwms(rng, 40)
    jobs = []
    for k in range(4):
        seqs = synth_seqs(rng, 120, 300, 800, p_n=0.002)
        cutoffs = cutoffs_for(pwms, seqs, 1e-3)
        jobs.append((seqs, cutoffs, oracle.scan_arrays(pwms, cutoffs, seqs, 3, n_threads=4)))
    ctx = eng.default_context(0)
    errors = []

    def work(seqs, cutoffs, expect):
        try:
            for _ in range(5):
                motifs = eng.MotifSet(ctx, pwms, cutoffs)
                sset = eng.SequenceSet(ctx, seqs)
                res = eng.scan(ctx, motifs, sset, 3)
                assert_scan_equal(res, expect)
                res.close(), sset.close(), motifs.close()
        except Exception as exc:   # noqa: BLE001
            errors.append(exc)

    threads = [threading.Thread(target=work, args=j) for j in jobs]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


def test_degenerate_shapes(eng):
    """Edges of the record path: only motifs the prefilter cannot take (L > 32), no motifs, no
    sequences, one 1-base sequence, empty result followed by the count accessors."""
    rng = np.random.default_rng(5)
    ctx = eng.default_context(0)
    seqs = synth_seqs(rng, 20, 100, 300, p_n=0.01)
    # (1) every motif longer than 32: the tensor-core prefilter has nothing to do
    slow = [rng.normal(0, 1.5, size=(4, L)).round(3).tolist() for L in (33, 40, 64)]
    cut = [0.2, 0.25, 0.1]
    motifs, sset = eng.MotifSet(ctx, slow, cut), eng.SequenceSet(ctx, seqs)
    res = eng.scan(ctx, motifs, sset, 3)
    assert_scan_equal(res, oracle.scan_arrays(slow, cut, seqs, 3, n_threads=4))
    assert res.n_sites > 0
    res.close(), motifs.close()
    # (2) no motifs
    none = eng.MotifSet(ctx, [], [])
    res = eng.scan(ctx, none, sset, 3)
    assert res.n_sites == 0 and len(res.counts) == 0
    res.close(), none.close(), sset.close()
    # (3) no sequences / one single base / only empty strings
    pwms = synth_pwms(rng, 5)
    motifs = eng.MotifSet(ctx, pwms, [0.5] * 5)
    for ss in ([], ["A"], ["", ""], ["N"]):
        sset = eng.SequenceSet(ctx, ss)
        res = eng.scan(ctx, motifs, sset, 3)
        assert res.n_sites == 0 and res.counts.tolist() == [0] * 5
        assert eng.scan_device(ctx, motifs, sset, 3) == 0
        assert ctx.site_counts(5).tolist() == [0] * 5 and ctx.region_counts(5).tolist() == [0] * 5
        a = eng.scan_ascii(ctx, motifs, *__import__("motifscan_b200")._lib.flatten_seqs(ss), 3)
        assert a.n_sites == 0
        a.close(), res.close(), sset.close()
    motifs.close()
