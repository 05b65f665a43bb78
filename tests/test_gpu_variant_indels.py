"""`motifscan variant --indels` on the GPU against an oracle built here, bit for bit.  Per allele the oracle trims REF
and ALT itself (longest common prefix, then suffix, bases compared as scoring sees them), splices the alt context on
the host, scans both contexts with `oracle.scan_arrays`, keeps the windows that touch the change (rules 4-5 of the
docs: s < c + k and s + L > c with k the side's changed length; paired when s < c + min(r', a') and the other window
fits) and scores a paired window on the other allele with `oracle.score_arrays`.  The indels are deletions and
insertions of 1 to more than Lmax bases on motifs of all three scan routes, complex alleles, at both chromosome ends,
into, out of and across an N run, inside a tandem repeat and on a chromosome shorter than the longest motif; one
motif has a cutoff of 0."""
import numpy as np
import pytest

import oracle
from motifscan_b200 import cli, engine, synth
from motifscan_b200 import io as msio
from motifscan_b200.genome import DeviceGenome, PackedGenome
from motifscan_b200.motif import MotifPwms, PositionWeightMatrix
from motifscan_b200.variants import read_vcf, scan_variants

pytestmark = pytest.mark.gpu
STRAND = {"+": 1, "-": 2, "both": 3}
BG = dict(A=0.295, C=0.205, G=0.205, T=0.295)
VCF_HEADER = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
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


def _bases(rng, k):
    return "".join(ACGT[i] for i in rng.integers(0, 4, k).tolist())


def _records(texts, rng):
    """(chrom, POS, ID, REF, ALT-field) records: the hard cases, then random indels, SNVs and MNVs."""
    recs = []

    def add(c, p, name, r, alt):                          # p 0-based, REF = r genome bases from p
        recs.append((c, p + 1, name, texts[c][p:p + r], alt))

    n1, n2, ns = len(texts["chr1"]), len(texts["chr2"]), len(texts["chrS"])
    t1 = texts["chr1"]
    for i, k in enumerate((1, 2, 5, 31, 33, 64, 65, 80)):  # deletions and insertions of 1 to more than Lmax bases
        p = 4200 + 300 * i
        add("chr1", p, f"del{k}", k + 1, t1[p])
        add("chr1", p + 150, f"ins{k}", 1, t1[p + 150] + _bases(rng, k))
    add("chr1", 6500, "cx1", 3, "GT")                       # complex alleles
    add("chr1", 6600, "cx2", 2, "TTACG")
    add("chr1", 6700, "cx3", 40, _bases(rng, 7))
    add("chr1", 0, "del_first", 4, t1[3])                  # chromosome starts: deletion / insertion at base 0
    add("chr1", 0, "ins_first", 1, _bases(rng, 6) + t1[0])
    add("chr2", n2 - 1, "ins_end", 1, texts["chr2"][-1] + _bases(rng, 30))   # after the last base: gains only
    add("chr2", n2 - 31, "del_end", 31, texts["chr2"][n2 - 31])               # reaches the end: unpaired losses
    add("chr1", n1 - 3, "cx_end", 3, "A")
    add("chr1", 1990, "del_intoN", 15, t1[1990])           # N run [2000, 2300): into, out of, across, inside
    add("chr1", 2290, "del_outofN", 20, "C")
    add("chr1", 1995, "del_acrossN", 320, t1[1995])
    add("chr1", 2100, "ins_inN", 1, "ACGTT")
    add("chr1", 1999, "ins_edgeN", 1, t1[1999] + "GATTACA")
    add("chr1", 1200, "del_repeat", 5, t1[1200])           # tandem repeat [1000, 1400)
    add("chr1", 1201, "ins_repeat", 1, t1[1201] + "TATA")
    add("chrS", 2, "del_short", 12, texts["chrS"][2])      # chromosome shorter than the longest motif
    add("chrS", 0, "del_whole", ns, "T")
    add("chrS", 9, "ins_short", 1, texts["chrS"][9] + _bases(rng, 25))
    add("chr1", 3100, "del_soft", 9, t1[3100].upper())     # soft-masked bases, REF in another case than ALT
    add("chr1", 7000, "multi", 1, f"{'C' if t1[7000].upper() != 'C' else 'G'},{t1[7000]}AAT,<DEL>")
    for k in range(90):
        c = "chr1" if k % 3 else "chr2"
        kind = k % 3
        n = len(texts[c])
        L = int(rng.integers(1, 50)) if k % 10 else int(rng.integers(70, 90))
        p = int(rng.integers(0, n - L - 2))
        if kind == 0:
            add(c, p, f"rd{k}", L + 1, texts[c][p])
        elif kind == 1:
            add(c, p, f"ri{k}", 1, texts[c][p] + _bases(rng, L))
        else:
            r = int(rng.integers(1, 4))
            add(c, p, f"rs{k}", r, _bases(rng, r))          # SNVs / MNVs (an occasional ALT == REF)
    add("chr1", 8000, "mnv", 3, "GAT")
    recs.append(("chrZ", 5, "unk", "A", "AG"))
    recs.append(("chr1", 3, "star", t1[2], "*"))
    return recs


def _write_vcf(path, recs):
    with open(path, "w") as fh:
        fh.write(VCF_HEADER + "".join(f"{c}\t{p}\t{i}\t{r}\t{a}\t.\tPASS\t.\n" for c, p, i, r, a in recs))


@pytest.fixture(scope="module")
def setup(tmp_path_factory):
    rng = np.random.default_rng(41)
    texts = {}
    for name, n in [("chr1", 9000), ("chr2", 3000), ("chrS", 20)]:
        s = bytearray(synth.random_bases(rng, n).tobytes())
        if n == 9000:
            s[1000:1400] = b"AT" * 200
            s[2000:2300] = b"N" * 300
            s[3000:3500] = bytes(s[3000:3500]).lower()
        texts[name] = bytes(s).decode()
    chroms = sorted(texts)
    packs = [synth.pack_ascii(np.frombuffer(texts[c].encode(), dtype=np.uint8)) for c in chroms]
    pg = PackedGenome(chroms, {c: len(texts[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                      np.concatenate([p[1] for p in packs]), name="ig")
    pwms = _pwms(rng, 18, 6, 30) + _pwms(rng, 4, 33, 40) + _pwms(rng, 2, 65, 70)
    cutoffs = _cutoffs(pwms, texts["chr1"][4100:] + texts["chr2"], rng)
    cutoffs[3] = 0.0
    recs = _records(texts, rng)
    root = tmp_path_factory.mktemp("indels")
    vcf = root / "calls.vcf"
    _write_vcf(vcf, recs)
    return dict(texts=texts, pg=pg, pwms=pwms, cutoffs=cutoffs, recs=recs, vcf=str(vcf),
                variants=read_vcf(str(vcf), pg, indels=True))


def _code(b):
    return ACGT.find(b.upper()) if b.upper() in ACGT else 4


def oracle_trim(ref, alt):
    """(offset of the change in REF, r', inserted bases); SNVs / MNVs untrimmed."""
    if len(ref) == len(alt):
        return 0, len(ref), alt
    m = min(len(ref), len(alt))
    pre = 0
    while pre < m and _code(ref[pre]) == _code(alt[pre]):
        pre += 1
    suf = 0
    while suf < m - pre and _code(ref[-1 - suf]) == _code(alt[-1 - suf]):
        suf += 1
    return pre, len(ref) - pre - suf, alt[pre:len(alt) - suf]


def oracle_rows(texts, v, pwms, cutoffs, strand):
    """Rows (allele, motif, haplotype start, strand, ref_score, alt_score, effect, paired), in the documented order."""
    lens = [len(p[0]) for p in pwms]
    lmax = max(lens)
    seqs, meta = [], []
    for a in range(len(v)):
        c = v.chroms[v.chrom[a]]
        pre, r, ins = oracle_trim(v.ref[a], v.alt[a])
        p = int(v.pos[a]) + pre
        cs, ce = max(p - lmax + 1, 0), min(p + r + lmax - 1, len(texts[c]))
        ref_ctx = texts[c][cs:ce]
        alt_ctx = ref_ctx[:p - cs] + ins + ref_ctx[p - cs + r:]
        seqs += [ref_ctx, alt_ctx]
        meta.append((cs, p - cs, r, len(ins)))
    counts, seq_idx, start, score, strd = oracle.scan_arrays(pwms, cutoffs, seqs, STRAND[strand], n_threads=8)
    motif_of = np.repeat(np.arange(len(pwms)), counts)
    hits = {}
    for m, q, s, sc, x in zip(motif_of.tolist(), seq_idx.tolist(), start.tolist(), score.tolist(), strd.tolist()):
        a, side = divmod(q, 2)
        cs, c0, r, k_alt = meta[a]
        k = k_alt if side else r
        if s >= c0 + k or s + lens[m] <= c0:
            continue
        paired = s < c0 + min(r, k_alt) and s + lens[m] <= len(seqs[2 * a + 1 - side])
        key = (a, m, s, x) if paired else (a, m, s, x, side)
        hits.setdefault(key, [None, None])[side] = sc
    todo = {}
    for key, sides in hits.items():
        if len(key) == 4:
            for side in (0, 1):
                if sides[side] is None:
                    a, m, s, x = key
                    todo.setdefault((m, x), []).append((key, side, seqs[2 * a + side][s:s + lens[m]]))
    for (m, x), items in todo.items():
        sc = oracle.score_arrays([pwms[m]], [w for _, _, w in items], x)[0]
        for (key, side, _), val in zip(items, sc.tolist()):
            hits[key][side] = val
    rows = []
    for key, (rs, al) in hits.items():
        a, m, s, x = key[:4]
        if len(key) == 5:
            rows.append((a, m, meta[a][0] + s, x, rs if rs is not None else np.nan, al if al is not None else np.nan,
                         1 if key[4] == 0 else 2, False))
            continue
        ref_hit, alt_hit = rs - cutoffs[m] >= -1e-10, al - cutoffs[m] >= -1e-10
        rows.append((a, m, meta[a][0] + s, x, rs, al, 3 if ref_hit and alt_hit else (1 if ref_hit else 2), True))
    rows.sort(key=lambda t: t[:4])
    return rows


def assert_rows(sites, rows):
    cols = list(zip(*rows)) if rows else [[]] * 8
    assert len(sites) == len(rows)
    assert np.array_equal(sites.allele, np.array(cols[0], np.int32))
    assert np.array_equal(sites.motif, np.array(cols[1], np.int32))
    assert np.array_equal(sites.start, np.array(cols[2], np.int64))
    assert np.array_equal(sites.strand, np.array(cols[3], np.int8))
    assert np.array_equal(sites.paired, np.array(cols[7], bool))
    for got, want in ((sites.ref_score, cols[4]), (sites.alt_score, cols[5])):
        want = np.array(want, np.float64)
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(got), nan)
        assert np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64))
    assert np.array_equal(sites.effect, np.array(cols[6], np.int8))


def test_extract_splice_equals_host_splice(setup):
    texts, v, pg = setup["texts"], setup["variants"], setup["pg"]
    ctx = engine.Context(0)
    dg = DeviceGenome(pg, ctx=ctx)
    try:
        n = len(v)
        idx = np.array([dg.chrom_index[v.chroms[c]] for c in v.chrom], dtype=np.int32)
        size = np.array([pg.chrom_sizes[v.chroms[c]] for c in v.chrom])
        trims = [oracle_trim(v.ref[a], v.alt[a]) for a in range(n)]
        p = np.array([int(v.pos[a]) + t[0] for a, t in enumerate(trims)])
        r = np.array([t[1] for t in trims])
        rng = np.random.default_rng(5)
        lo, hi = rng.integers(0, 40, n), rng.integers(0, 40, n)
        lo[:3], hi[:3] = 0, 0                                   # contexts of exactly the deleted bases
        cs = np.maximum(p - lo, 0)
        ce = np.minimum(p + r + hi, size)
        ins = [t[2] for t in trims]
        for k in range(3):
            ins[k] = ""                                          # pure deletions of the whole context: empty
        ins_off = np.concatenate([[0], np.cumsum([len(x) for x in ins])])
        ins_code = np.array([ACGT.index(b) for b in "".join(ins).upper()], dtype=np.uint8)
        alt = dg.seqs.extract_splice(idx, cs, ce, p - cs, r, ins_off, ins_code)
        want = []
        for a in range(n):
            t = texts[v.chroms[v.chrom[a]]][cs[a]:ce[a]]
            want.append(t[:p[a] - cs[a]] + ins[a] + t[p[a] - cs[a] + r[a]:])
        assert sum(len(w) == 0 for w in want) >= 3
        assert np.array_equal(alt.codes(), np.concatenate([oracle.encode(w) for w in want]))
        alt.close()
        empty = dg.seqs.extract_splice(idx[:0], cs[:0], ce[:0], [], [], [0], [])
        assert empty.n == 0
        empty.close()
        span = int(ce[5] - cs[5])
        for at, dl, off, code in ((span, 1, [0, 0], []), (-1, 0, [0, 1], [0]), (0, span + 1, [0, 0], []),
                                  (0, 0, [0, 1], [4]), (0, 0, [1, 1], []), (0, -1, [0, 0], [])):
            with pytest.raises(ValueError):
                dg.seqs.extract_splice(idx[5:6], cs[5:6], ce[5:6], [at], [dl], off, np.array(code, dtype=np.uint8))
    finally:
        dg.close()
        ctx.close()


@pytest.mark.parametrize("strand", ["+", "-", "both"])
def test_rows_equal_oracle(setup, strand):
    v = setup["variants"]
    rows = oracle_rows(setup["texts"], v, setup["pwms"], setup["cutoffs"], strand)
    sites = scan_variants(setup["pg"], setup["pwms"], setup["cutoffs"], v, strand=strand)
    assert_rows(sites, rows)
    if strand == "both":
        assert sites.paired.any() and (~sites.paired & (sites.effect == 1)).any() and (~sites.paired & (sites.effect == 2)).any()
        ids = np.array(v.id)[sites.allele]
        assert (ids == "ins_end").any() and (sites.effect[ids == "ins_end"] == 2).all() and not sites.paired[ids == "ins_end"].any()
        assert (ids == "del_end").any() and (~sites.paired[(ids == "del_end") & (sites.effect == 1)]).any()
        assert (sites.motif >= 22).any() and (sites.motif[~sites.paired] >= 18).any()
        assert (sites.motif == 3).any()
        n_indel = sum(len(a) != len(r) for a, r in zip(v.alt, v.ref))
        bad_alt = sum(not set(a) <= set("ACGTacgt") for *_, alts in setup["recs"] for a in alts.split(","))
        assert n_indel > 60 and v.skipped["unsupported"] == bad_alt >= 2 and v.skipped["unknown_chrom"] == 1


def test_overflow_retry_keeps_rows(setup):
    rows = oracle_rows(setup["texts"], setup["variants"], setup["pwms"], setup["cutoffs"], "both")
    ctx = engine.Context(0)
    dg = DeviceGenome(setup["pg"], ctx=ctx)
    try:
        ctx.set_option("tc_first_lane_cap", 1)
        sites = scan_variants(dg, setup["pwms"], setup["cutoffs"], setup["variants"])
        assert ctx.counters()["retries"] > 0
        assert_rows(sites, rows)
    finally:
        dg.close()
        ctx.close()


def test_snv_mnv_rows_equal_default_mode(setup):
    v = setup["variants"]
    d = read_vcf(setup["vcf"], setup["pg"])
    assert not d.indels and 0 < len(d) < len(v)
    both = scan_variants(setup["pg"], setup["pwms"], setup["cutoffs"], v)
    plain = scan_variants(setup["pg"], setup["pwms"], setup["cutoffs"], d)
    same_len = np.flatnonzero([len(a) == len(r) for a, r in zip(v.alt, v.ref)])
    assert [v.id[a] for a in same_len] == d.id
    new_index = np.full(len(v), -1)
    new_index[same_len] = np.arange(len(same_len))
    sel = new_index[both.allele] >= 0
    assert sel.sum() == len(plain) > 0 and both.paired[sel].all()
    assert np.array_equal(new_index[both.allele[sel]], plain.allele)
    for name in ("motif", "start", "strand", "effect"):
        assert np.array_equal(getattr(both, name)[sel], getattr(plain, name))
    for name in ("ref_score", "alt_score"):
        assert np.array_equal(getattr(both, name)[sel].view(np.uint64), getattr(plain, name).view(np.uint64))


def _render(v, back, rows):
    names = {1: "loss", 2: "gain", 3: "both"}
    out = msio.VARIANT_SITES_HEADER
    for a, m, s, x, rs, al, e, paired in rows:
        rt = "NA" if not paired and e == 2 else str(rs)
        at = "NA" if not paired and e == 1 else str(al)
        out += (f"{v.chroms[v.chrom[a]]}\t{v.pos[a] + 1}\t{v.id[a]}\t{v.ref[a]}\t{v.alt[a]}\t{back[m].matrix_id}\t"
                f"{back[m].name}\t{s}\t{s + back[m].length}\t{'+' if x == 1 else '-'}\t{rt}\t{at}\t{names[e]}\n")
    summ = msio.VARIANT_SUMMARY_HEADER
    for m, p in enumerate(back):
        n = [len({r[0] for r in rows if r[1] == m and r[6] == e}) for e in (2, 1, 3)]
        summ += f"{p.matrix_id}\t{p.name}\t{n[0]}\t{n[1]}\t{n[2]}\n"
    return out, summ


def test_cli_tables_equal_oracle(setup, tmp_path):
    gdir, mdir = tmp_path / "ig", tmp_path / "im"
    gdir.mkdir(), mdir.mkdir()
    with open(gdir / "ig.fa", "w") as fh:
        for c in sorted(setup["texts"]):
            t = setup["texts"][c]
            fh.write(f">{c}\n" + "".join(t[i:i + 60] + "\n" for i in range(0, len(t), 60)))
    pw = MotifPwms(name="im", genome="ig")
    for k, (m, c) in enumerate(zip(setup["pwms"], setup["cutoffs"])):
        pw.append(PositionWeightMatrix(np.array(m), name=f"TF{k}", matrix_id=f"MA{k:04d}.1", cutoffs={"1e-4": c}))
    pw.write_motifscan_pwms(str(mdir / "im_ig_pwms.motifscan"))
    back = MotifPwms()
    back.read_motifscan_pwms(str(mdir / "im_ig_pwms.motifscan"))
    pwms, cutoffs = [p.matrix for p in back], [p.cutoffs["1e-4"] for p in back]
    for flag, v in ((["--indels"], setup["variants"]), ([], read_vcf(setup["vcf"], setup["pg"]))):
        out = tmp_path / f"out{len(flag)}"
        assert cli.main(["variant", "-i", setup["vcf"], "-m", str(mdir), "-g", str(gdir), "-o", str(out)] + flag) == 0
        rows = oracle_rows(setup["texts"], v, pwms, cutoffs, "both")
        assert any(not r[7] for r in rows) == bool(flag)
        sites, summ = _render(v, back, rows)
        assert (out / "motif_variant_sites.xls").read_text() == sites
        assert (out / "motif_variant_summary.xls").read_text() == summ
