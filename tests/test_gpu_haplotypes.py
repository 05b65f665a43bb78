"""`motifscan variant --haplotypes` on the GPU against an oracle built here, bit for bit.  Per cluster the oracle
applies every allele's change to the reference context on the host, keeping a per-base origin map of the alt string
(the ref base each alt base came from: a flank base, or a core base at an offset below min(r', a'); -1 otherwise),
scans both strings with `oracle.scan_arrays`, finds the affected windows from the core bases and junctions of each
side, pairs windows through the origin map and scores a paired window on the other side with `oracle.score_arrays`.
It emits a row for every pair in which an affected window is a site, without assuming that paired windows are
affected together.  Clusters: two SNVs that make or break a site only together, an SNV next to a deletion, a deletion
followed by an insertion, a dense cluster of 40+ edits, clusters at both chromosome ends, into and across an N run, in
a tandem repeat, on a 20-base chromosome (one with an empty alt context), and random ones; motifs on all three scan
routes, one with a cutoff of 0."""
import numpy as np
import pytest

import oracle
from motifscan_b200 import cli, engine, synth
from motifscan_b200 import io as msio
from motifscan_b200.genome import DeviceGenome, PackedGenome
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
from motifscan_b200.variants import haplotype_clusters, read_vcf, scan_haplotypes, scan_variants

pytestmark = pytest.mark.gpu
STRAND = {"+": 1, "-": 2, "both": 3}
BG = dict(A=0.295, C=0.205, G=0.205, T=0.295)
ACGT = "ACGT"


def _pwms(rng, n, lmin, lmax):
    out = []
    for _ in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        pfm = np.round(int(rng.integers(20, 3000)) * rng.dirichlet([0.3] * 4, size=L).T).astype(np.int64)
        pfm[0, pfm.sum(axis=0) == 0] = 1
        out.append(oracle.pfm_to_pwm(pfm, BG).tolist())
    return out


def _cutoffs(pwms, text, rng, rate=4e-3):
    lmax = max(len(p[0]) for p in pwms)
    starts = rng.integers(0, len(text) - lmax, 3000)
    samples = [text[a:a + lmax].upper().replace("N", "A") for a in starts.tolist()]
    sc = oracle.score_arrays(pwms, samples, 3)
    k = max(int(len(samples) * rate), 1)
    return [float(np.sort(row)[::-1][k]) for row in sc]


def _other(b, rng):
    return ACGT[(ACGT.index(b.upper()) + int(rng.integers(1, 4))) % 4] if b.upper() in ACGT else "A"


def _plant(text, pwm, at):
    """Write the motif's best bases at `at`; returns the text and the window."""
    best = "".join(ACGT[int(np.argmax(col))] for col in np.array(pwm).T)
    return text[:at] + best + text[at + len(best):], best


def _groups(texts, rng, planted):
    """Haplotype groups: lists of (chrom, 0-based POS, REF, ALT, ID) records carried together on one haplotype."""
    t1, t2, tS = texts["chr1"], texts["chr2"], texts["chrS"]
    n1, n2 = len(t1), len(t2)
    g = []

    def snv(c, p, alt=None, name=None):
        t = texts[c]
        return (c, p, t[p], alt or _other(t[p], rng), name or f"s{c}_{p}")

    def dele(c, p, k, name=None):                   # removes [p, p + k), anchored at p - 1
        t = texts[c]
        return (c, p - 1, t[p - 1:p + k], t[p - 1], name or f"d{c}_{p}_{k}")

    def ins(c, p, bases, name=None):                # inserts before base p, anchored at p - 1
        t = texts[c]
        return (c, p - 1, t[p - 1], t[p - 1] + bases, name or f"i{c}_{p}_{len(bases)}")

    def bases(k):
        return "".join(ACGT[i] for i in rng.integers(0, 4, k).tolist())

    # planted pairs (motif 0's best window at 5000, and at 5600 with bases i and j changed): the break pair and the
    # make pair with their singletons
    (i, bi, best_i), (j, bj, best_j), best = planted
    brk = [("chr1", 5000 + i, best_i, bi, "brk_i"), ("chr1", 5000 + j, best_j, bj, "brk_j")]
    g += [brk, brk[:1], brk[1:]]
    mk = [("chr1", 5600 + i, bi, best_i, "mk_i"), ("chr1", 5600 + j, bj, best_j, "mk_j")]
    g += [mk, mk[:1]]
    g.append([snv("chr1", 4199, name="snv_gap0"), dele("chr1", 4200, 6, name="del_gap0")])        # gap 0
    # a deletion [4400, 4403), then motif 0's best window inserted at 4410 while the reference has it at 4407: the
    # reference site at 4407 straddles the insertion's junction and the inserted copy starts at 4410 - 3 = 4407 on
    # the haplotype, an unpaired gain -- a ref row and an alt row at the same (start, strand)
    g.append([dele("chr1", 4400, 3, name="del_then"), ins("chr1", 4410, best, name="then_ins")])
    dense, p = [], 6000                              # 40+ edits in ~100 bp
    while p < 6100:
        kind = int(rng.integers(0, 6))
        if kind == 0:
            k = int(rng.integers(1, 3))
            dense.append(dele("chr1", p, k))
            p += k
        elif kind == 1:
            dense.append(ins("chr1", p, bases(int(rng.integers(1, 4)))))
            p += 1
        else:
            dense.append(snv("chr1", p))
            p += 1
        p += int(rng.integers(0, 2))
    assert len(dense) >= 40
    g.append(dense)
    g.append([(("chr1", 0, t1[0], bases(5) + t1[0], "ins_first")), snv("chr1", 2, name="s_first")])   # chromosome starts
    g.append([snv("chr2", n2 - 3, name="s_end"), ("chr2", n2 - 1, t2[-1], t2[-1] + bases(12), "ins_end")])
    g.append([snv("chr2", n2 - 40, name="s_end2"), dele("chr2", n2 - 30, 30, name="del_end")])
    g.append([snv("chr1", 1985, name="s_intoN"), dele("chr1", 1995, 15, name="del_intoN")])      # N run [2000, 2300)
    g.append([snv("chr1", 1990, name="s_acrossN"), dele("chr1", 1996, 310, name="del_acrossN"), snv("chr1", 2310)])
    g.append([ins("chr1", 2000, "ACGTT", name="ins_edgeN"), ("chr1", 2099, "N", "GACGTT", "cx_inN"),
              ("chr1", 2105, "N", "G", "n_to_g")])
    g.append([dele("chr1", 1200, 2, name="del_rep"), snv("chr1", 1205), ins("chr1", 1210, "TA", name="ins_rep")])
    # chrS (20 bases): deleting [0, 9) and [9, 20) leaves an empty alt context
    g.append([("chrS", 0, tS[0:10], tS[9], "del_s0"), ("chrS", 8, tS[8:20], tS[8], "del_s1")])
    g.append([snv("chrS", 3, name="s_short"), ins("chrS", 10, bases(25), name="ins_short")])
    for k in range(40):                              # random clusters of 2-5 alleles within ~30 bp
        c = "chr1" if k % 3 else "chr2"
        t = texts[c]
        p = int(rng.integers(2500, len(t) - 100)) if c == "chr1" else int(rng.integers(10, len(t) - 100))
        grp = []
        for _ in range(int(rng.integers(2, 6))):
            kind = int(rng.integers(0, 4))
            if kind == 0:
                grp.append(snv(c, p))
                p += 1
            elif kind == 1:
                k_ = int(rng.integers(1, 40))
                grp.append(dele(c, p, k_))
                p += k_
            elif kind == 2:
                grp.append(ins(c, p, bases(int(rng.integers(1, 40)))))
            else:
                grp.append((c, p, t[p:p + 2], bases(2), f"m{c}_{p}"))
                p += 2
            p += int(rng.integers(1, 8))
        g.append(grp)
    for k in range(24):                              # singletons: SNVs, MNVs, deletions and insertions on their own
        c = "chr1" if k % 2 else "chr2"
        p = int(rng.integers(2500, n1 - 100)) if c == "chr1" else int(rng.integers(10, n2 - 100))
        kind = k % 4
        g.append([snv(c, p) if kind == 0 else dele(c, p, int(rng.integers(1, 40))) if kind == 1 else
                  ins(c, p, bases(int(rng.integers(1, 40)))) if kind == 2 else (c, p, texts[c][p:p + 3], bases(3), f"m{c}_{p}")])
    return g


def _vcf(path, groups, chroms):
    """A phased VCF: group k is haplotype k % 2 of sample k // 2 (plus S_ref, homozygous reference)."""
    recs = {}
    for k, grp in enumerate(groups):
        for r in grp:
            recs.setdefault(r, set()).add(k)
    n_s = (len(groups) + 1) // 2
    names = [f"S{i}" for i in range(n_s)] + ["S_ref"]
    order = sorted(recs, key=lambda r: (chroms.index(r[0]), r[1], r[2], r[3]))
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(names) + "\n")
        for r in order:
            gts = [f"{int(2 * s in recs[r])}|{int(2 * s + 1 in recs[r])}" for s in range(n_s)] + ["0|0"]
            fh.write(f"{r[0]}\t{r[1] + 1}\t{r[4]}\t{r[2]}\t{r[3]}\t.\tPASS\t.\tGT\t" + "\t".join(gts) + "\n")
    return names


@pytest.fixture(scope="module")
def setup(tmp_path_factory):
    rng = np.random.default_rng(43)
    texts = {}
    for name, n in [("chr1", 9000), ("chr2", 3000), ("chrS", 20)]:
        s = bytearray(synth.random_bases(rng, n).tobytes())
        if n == 9000:
            s[1000:1400] = b"AT" * 200
            s[2000:2300] = b"N" * 300
            s[3000:3500] = bytes(s[3000:3500]).lower()
        if n == 20:
            s[0], s[9] = ord("A"), ord("C")          # the two deletions' trimming stays as built
        texts[name] = bytes(s).decode()
    pwms = _pwms(rng, 18, 6, 30) + _pwms(rng, 4, 33, 40) + _pwms(rng, 2, 65, 70)
    cutoffs = _cutoffs(pwms, texts["chr1"][4100:] + texts["chr2"], rng)
    cutoffs[3] = 0.0
    # planted: motif 0's best window at 5000 (the break pair), with two bases changed at 5600 (the make pair), and at
    # 4407 (the deletion-then-insertion case); motif 24 / 25 are motif 0 with cutoffs between the scores of the window
    # with none, one and both bases changed
    t1, best = _plant(texts["chr1"], pwms[0], 5000)
    L0, i, j = len(best), 3, 9
    assert L0 > 3                                    # the window at 4407 reaches the junction at 4410
    bi = ACGT[int(np.argmin(np.array(pwms[0])[:, i]))]
    bj = ACGT[int(np.argmin(np.array(pwms[0])[:, j]))]
    variants_ = [best, best[:i] + bi + best[i + 1:], best[:j] + bj + best[j + 1:],
                 best[:i] + bi + best[i + 1:j] + bj + best[j + 1:]]
    sc = oracle.score_arrays([pwms[0]], variants_, 1)[0]
    assert sc[3] < min(sc[1], sc[2]) and max(sc[1], sc[2]) < sc[0]
    t1 = t1[:5600] + variants_[3] + t1[5600 + L0:]
    t1 = t1[:4407] + best + t1[4407 + L0:]
    texts["chr1"] = t1
    pwms += [pwms[0], pwms[0]]
    cutoffs += [float((sc[3] + min(sc[1], sc[2])) / 2), float((max(sc[1], sc[2]) + sc[0]) / 2)]
    chroms = sorted(texts)
    packs = [synth.pack_ascii(np.frombuffer(texts[c].encode(), dtype=np.uint8)) for c in chroms]
    pg = PackedGenome(chroms, {c: len(texts[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                      np.concatenate([p[1] for p in packs]), name="hg")
    groups = _groups(texts, rng, ((i, bi, best[i]), (j, bj, best[j]), best))
    root = tmp_path_factory.mktemp("haps")
    vcf = str(root / "phased.vcf")
    _vcf(vcf, groups, chroms)
    v = read_vcf(vcf, pg, indels=True, samples="all")
    lmax = max(len(p[0]) for p in pwms)
    return dict(texts=texts, pg=pg, pwms=pwms, cutoffs=cutoffs, vcf=vcf, variants=v, haps=haplotype_clusters(v, lmax))


def _code(b):
    return ACGT.find(b.upper()) if b.upper() in ACGT else 4


def oracle_change(ref, alt, indels):
    """(offset of the change in REF, r', inserted bases); SNVs / MNVs untrimmed."""
    if len(ref) == len(alt) or not indels:
        return 0, len(ref), alt
    m = min(len(ref), len(alt))
    pre = 0
    while pre < m and _code(ref[pre]) == _code(alt[pre]):
        pre += 1
    suf = 0
    while suf < m - pre and _code(ref[-1 - suf]) == _code(alt[-1 - suf]):
        suf += 1
    return pre, len(ref) - pre - suf, alt[pre:len(alt) - suf]


def oracle_contexts(texts, h, lmax):
    """Per cluster: (cs, ref string, alt string, origin map, ref core mask, alt core mask, ref / alt junctions)."""
    v = h.variants
    out = []
    for c in range(len(h)):
        t = texts[v.chroms[h.chrom[c]]]
        ch = []
        for a in h.allele[h.allele_off[c]:h.allele_off[c + 1]].tolist():
            pre, r, ins = oracle_change(v.ref[a], v.alt[a], v.indels)
            ch.append((int(v.pos[a]) + pre, r, ins))
        cs = max(ch[0][0] - lmax + 1, 0)
        ce = min(ch[-1][0] + ch[-1][1] + lmax - 1, len(t))
        ref = t[cs:ce]
        alt, origin, alt_core, ref_core, ref_j, alt_j = "", [], [], np.zeros(len(ref), bool), set(), set()
        prev = 0
        for p, r, ins in ch:
            q = p - cs
            alt += ref[prev:q]
            origin += list(range(prev, q))
            alt_core += [False] * (q - prev)
            if not ins:
                alt_j.add(len(alt))
            if r == 0:
                ref_j.add(q)
            ref_core[q:q + r] = True
            for o in range(len(ins)):
                origin.append(q + o if o < min(r, len(ins)) else -1)
                alt_core.append(True)
            alt += ins
            prev = q + r
        alt += ref[prev:]
        origin += list(range(prev, len(ref)))
        alt_core += [False] * (len(ref) - prev)
        out.append((cs, ref, alt, np.array(origin, np.int64), ref_core, np.array(alt_core, bool), ref_j, alt_j))
    return out


def _affected(core, junctions, s, L):
    return bool(core[s:s + L].any()) or any(s < j < s + L for j in junctions)


def oracle_rows(texts, h, pwms, cutoffs, strand):
    """Rows (cluster, motif, strand, ref_start, alt_start, ref_score, alt_score, effect, paired) in the documented
    order (cluster, motif, own-side start, strand, ref before alt)."""
    lens = [len(p[0]) for p in pwms]
    ctxs = oracle_contexts(texts, h, max(lens))
    seqs = [x for cx in ctxs for x in (cx[1], cx[2])]
    counts, seq_idx, start, score, strd = oracle.scan_arrays(pwms, cutoffs, seqs, STRAND[strand], n_threads=8)
    motif_of = np.repeat(np.arange(len(pwms)), counts)
    inv = []
    for cx in ctxs:
        m = np.full(len(cx[1]) + 1, -1, np.int64)
        ok = cx[3] >= 0
        m[cx[3][ok]] = np.flatnonzero(ok)
        inv.append(m)
    pairs, rows = {}, []
    for m, q, s, sc, x in zip(motif_of.tolist(), seq_idx.tolist(), start.tolist(), score.tolist(), strd.tolist()):
        c, side = divmod(q, 2)
        cs, ref, alt, origin, ref_core, alt_core, ref_j, alt_j = ctxs[c]
        L = lens[m]
        if side == 0:
            if not _affected(ref_core, ref_j, s, L):
                continue
            t = int(inv[c][s])
            if t >= 0 and t + L <= len(alt):
                pairs.setdefault((c, m, s, t, x), [None, None])[0] = sc
            else:
                rows.append((c, m, s, x, 0, cs + s, -1, sc, np.nan, 1, False))
        else:
            if not _affected(alt_core, alt_j, s, L):
                continue
            r = int(origin[s])
            if r >= 0 and r + L <= len(ref):
                pairs.setdefault((c, m, r, s, x), [None, None])[1] = sc
            else:
                rows.append((c, m, s, x, 1, -1, cs + s, np.nan, sc, 2, False))
    todo = {}
    for key, sides in pairs.items():
        c, m, s, t, x = key
        for side in (0, 1):
            if sides[side] is None:
                w = (ctxs[c][1][s:s + lens[m]], ctxs[c][2][t:t + lens[m]])[side]
                todo.setdefault((m, x), []).append((key, side, w))
    for (m, x), items in todo.items():
        sc = oracle.score_arrays([pwms[m]], [w for _, _, w in items], x)[0]
        for (key, side, _), val in zip(items, sc.tolist()):
            pairs[key][side] = val
    for (c, m, s, t, x), (rs, al) in pairs.items():
        ref_hit, alt_hit = rs - cutoffs[m] >= -1e-10, al - cutoffs[m] >= -1e-10
        eff = 3 if ref_hit and alt_hit else (1 if ref_hit else 2)
        cs = ctxs[c][0]
        rows.append((c, m, s if ref_hit else t, x, 0 if ref_hit else 1, cs + s, cs + t, rs, al, eff, True))
    rows.sort(key=lambda r: r[:5])
    return [(c, m, x, rs, at, a, b, e, p) for c, m, _, x, _, rs, at, a, b, e, p in rows]


def assert_rows(sites, rows):
    cols = list(zip(*rows)) if rows else [[]] * 9
    assert len(sites) == len(rows)
    for name, k, dt in (("cluster", 0, np.int32), ("motif", 1, np.int32), ("strand", 2, np.int8),
                        ("ref_start", 3, np.int64), ("alt_start", 4, np.int64), ("effect", 7, np.int8), ("paired", 8, bool)):
        assert np.array_equal(getattr(sites, name), np.array(cols[k], dt)), name
    for got, want in ((sites.ref_score, cols[5]), (sites.alt_score, cols[6])):
        want = np.array(want, np.float64)
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(got), nan)
        assert np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64))


def _cluster_of(h, ids):
    v = h.variants
    want = set(ids)
    for c in range(len(h)):
        if {v.id[a] for a in h.allele[h.allele_off[c]:h.allele_off[c + 1]].tolist()} == want:
            return c
    raise AssertionError(f"no cluster {ids}")


def test_extract_edits_equals_host_strings(setup):
    h, pg, texts = setup["haps"], setup["pg"], setup["texts"]
    lmax = max(len(p[0]) for p in setup["pwms"])
    ctxs = oracle_contexts(texts, h, lmax)
    assert any(len(cx[2]) == 0 for cx in ctxs) and h.sizes().max() >= 40
    ctx = engine.Context(0)
    dg = DeviceGenome(pg, ctx=ctx)
    try:
        v = h.variants
        idx = np.array([dg.chrom_index[v.chroms[c]] for c in h.chrom], dtype=np.int32)
        cs = np.array([cx[0] for cx in ctxs])
        ce = cs + np.array([len(cx[1]) for cx in ctxs])
        al = h.allele
        ch = [oracle_change(v.ref[a], v.alt[a], True) for a in al.tolist()]
        at = np.array([int(v.pos[a]) + c[0] for a, c in zip(al.tolist(), ch)]) - np.repeat(cs, h.sizes())
        dl = np.array([c[1] for c in ch])
        ins_off = np.concatenate([[0], np.cumsum([len(c[2]) for c in ch])])
        code = np.array([ACGT.index(b.upper()) for c in ch for b in c[2]], dtype=np.uint8)
        alt = dg.seqs.extract_edits(idx, cs, ce, h.allele_off, at, dl, ins_off, code)
        assert np.array_equal(alt.codes(), np.concatenate([oracle.encode(cx[2]) for cx in ctxs]))
        alt.close()
        # each validation error is MSB_EINVAL (ValueError): out of order, overlapping, outside, a code above 3
        k = int(np.argmax(ce - cs >= 20))
        one = lambda a, d, c: dg.seqs.extract_edits(idx[k:k + 1], cs[k:k + 1], ce[k:k + 1], [0, 3], a, d,   # noqa: E731
                                                    [0, 1, 2, 3], np.array(c, dtype=np.uint8))
        one(np.array([0, 2, 4]), [1, 1, 1], [0, 1, 2]).close()
        for a, d, c in (([4, 2, 6], [1, 1, 1], [0, 1, 2]), ([0, 1, 4], [2, 1, 1], [0, 1, 2]),
                        ([0, 0, 4], [0, 1, 1], [0, 1, 2]), ([0, 2, int(ce[k] - cs[k])], [1, 1, 1], [0, 1, 2]),
                        ([0, 2, 4], [1, 1, 1], [0, 4, 2]), ([-1, 2, 4], [1, 1, 1], [0, 1, 2])):
            with pytest.raises(ValueError):
                one(np.array(a), d, c)
    finally:
        dg.close()
        ctx.close()


@pytest.mark.parametrize("strand", ["+", "-", "both"])
def test_rows_equal_oracle(setup, strand):
    h = setup["haps"]
    rows = oracle_rows(setup["texts"], h, setup["pwms"], setup["cutoffs"], strand)
    sites = scan_haplotypes(setup["pg"], setup["pwms"], setup["cutoffs"], h, strand=strand)
    assert_rows(sites, rows)
    if strand != "both":
        return
    # the planted pairs: breaking (motif 24) and making (motif 25) a site only together
    for ids, m, want in ((("brk_i", "brk_j"), 24, 1), (("mk_i", "mk_j"), 25, 2)):
        both = _cluster_of(h, ids)
        sel = (sites.cluster == both) & (sites.motif == m) & (sites.effect == want) & (sites.strand == 1)
        hit = set(sites.ref_start[sel].tolist())
        assert (5000 if want == 1 else 5600) in hit
        one = _cluster_of(h, ids[:1])
        sel1 = (sites.cluster == one) & (sites.motif == m) & (sites.strand == 1)
        assert (5000 if want == 1 else 5600) not in set(sites.ref_start[sel1 & (sites.effect == want)].tolist())
    # a deletion then an insertion: a ref row and an alt row share (start, strand)
    c = _cluster_of(h, ("del_then", "then_ins"))
    sel = sites.cluster == c
    own = np.where(sites.effect == 2, sites.alt_start, sites.ref_start)
    keys = {}
    for m, s, x, e in zip(sites.motif[sel].tolist(), own[sel].tolist(), sites.strand[sel].tolist(), sites.effect[sel].tolist()):
        keys.setdefault((m, s, x), set()).add(e == 2)
    assert any(len(k) == 2 for k in keys.values())
    assert (~sites.paired & (sites.effect == 1)).any() and (~sites.paired & (sites.effect == 2)).any()
    assert (sites.motif >= 22).any() and (sites.motif == 3).any()


def test_overflow_retry_keeps_rows(setup):
    rows = oracle_rows(setup["texts"], setup["haps"], setup["pwms"], setup["cutoffs"], "both")
    ctx = engine.Context(0)
    dg = DeviceGenome(setup["pg"], ctx=ctx)
    try:
        ctx.set_option("tc_first_lane_cap", 1)
        sites = scan_haplotypes(dg, setup["pwms"], setup["cutoffs"], setup["haps"])
        assert ctx.counters()["retries"] > 0
        assert_rows(sites, rows)
    finally:
        dg.close()
        ctx.close()


@pytest.mark.parametrize("indels", [True, False])
def test_singleton_clusters_reproduce_scan_variants(setup, indels):
    v = read_vcf(setup["vcf"], setup["pg"], indels=indels, samples="all")
    h = haplotype_clusters(v, max(len(p[0]) for p in setup["pwms"]))
    single = np.flatnonzero(h.sizes() == 1)
    assert len(single) > 10
    hs = scan_haplotypes(setup["pg"], setup["pwms"], setup["cutoffs"], h)
    vs = scan_variants(setup["pg"], setup["pwms"], setup["cutoffs"], v)
    cl_of = np.full(len(v), -1)
    cl_of[h.allele[h.allele_off[single]]] = single
    vsel = np.flatnonzero(cl_of[vs.allele] >= 0)
    vsel = vsel[np.argsort(cl_of[vs.allele[vsel]], kind="stable")]
    hsel = np.flatnonzero(np.isin(hs.cluster, single))
    assert len(hsel) == len(vsel) > 0
    assert np.array_equal(hs.cluster[hsel], cl_of[vs.allele[vsel]])
    for name in ("motif", "strand", "effect", "paired"):
        assert np.array_equal(getattr(hs, name)[hsel], getattr(vs, name)[vsel]), name
    for name in ("ref_score", "alt_score"):
        assert np.array_equal(getattr(hs, name)[hsel].view(np.uint64), getattr(vs, name)[vsel].view(np.uint64))
    own = np.where(hs.effect[hsel] == 2, hs.alt_start[hsel], hs.ref_start[hsel])
    assert np.array_equal(own, vs.start[vsel])


def _motif_dirs(setup, tmp_path):
    gdir, mdir = tmp_path / "hg", tmp_path / "im"
    gdir.mkdir(), mdir.mkdir()
    with open(gdir / "hg.fa", "w") as fh:
        for c in sorted(setup["texts"]):
            t = setup["texts"][c]
            fh.write(f">{c}\n" + "".join(t[i:i + 60] + "\n" for i in range(0, len(t), 60)))
    pw = MotifPwms(name="im", genome="hg")
    for k, (m, c) in enumerate(zip(setup["pwms"], setup["cutoffs"])):
        pw.append(PositionWeightMatrix(np.array(m), name=f"TF{k}", matrix_id=f"MA{k:04d}.1", cutoffs={"1e-4": c}))
    pw.write_motifscan_pwms(str(mdir / "im_hg_pwms.motifscan"))
    back = MotifPwms()
    back.read_motifscan_pwms(str(mdir / "im_hg_pwms.motifscan"))
    return gdir, mdir, back


def test_cli_tables_equal_written_tables(setup, tmp_path):
    gdir, mdir, back = _motif_dirs(setup, tmp_path)
    pwms, cutoffs = [p.matrix for p in back], [p.cutoffs["1e-4"] for p in back]
    out = tmp_path / "out"
    assert cli.main(["variant", "-i", setup["vcf"], "-m", str(mdir), "-g", str(gdir), "-o", str(out), "--indels",
                     "--haplotypes"]) == 0
    assert sorted(p.name for p in out.iterdir()) == ["motif_haplotype_clusters.xls", "motif_haplotype_sites.xls",
                                                     "motif_haplotype_summary.xls"]
    h = setup["haps"]
    sites = scan_haplotypes(setup["pg"], pwms, cutoffs, h)
    assert_rows(sites, oracle_rows(setup["texts"], h, pwms, cutoffs, "both"))
    want = tmp_path / "want"
    msio.write_haplotype_tables(str(want), back, h, sites)
    for name in ("motif_haplotype_sites.xls", "motif_haplotype_clusters.xls", "motif_haplotype_summary.xls"):
        assert (out / name).read_bytes() == (want / name).read_bytes(), name
    # only the homozygous-reference sample: header-only tables
    ref_only = tmp_path / "ref_only"
    assert cli.main(["variant", "-i", setup["vcf"], "-m", str(mdir), "-g", str(gdir), "-o", str(ref_only),
                     "--haplotypes", "--samples", "S_ref"]) == 0
    assert (ref_only / "motif_haplotype_sites.xls").read_text() == msio.HAPLOTYPE_SITES_HEADER
    assert (ref_only / "motif_haplotype_clusters.xls").read_text() == msio.HAPLOTYPE_CLUSTERS_HEADER
    summ = (ref_only / "motif_haplotype_summary.xls").read_text().splitlines()
    assert len(summ) == len(back) + 1 and all(line.endswith("\t0\t0\t0\t0\t0\t0") for line in summ[1:])
