"""`motifscan variant` on the GPU against an oracle built here, bit for bit: per allele, the ref and alt context
strings are built on the host and scanned with `oracle.scan_arrays`; the windows that overlap the changed bases are
kept, and the window's score on the other allele comes from `oracle.score_arrays` on its L bases.  The genome holds
N runs, soft-masked runs, a tandem repeat and a chromosome shorter than the longest motif; the variants sit at
chromosome ends, next to each other, several at one position, across N runs and with ALT == REF; the motifs take
all three scan routes (<= 32, 33-64 and > 64 columns), one has a cutoff of 0 and two have cutoffs that equal window
scores exactly."""
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


def _pwms(rng, n, lmin, lmax):
    out = []
    for _ in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        pfm = np.round(int(rng.integers(20, 3000)) * rng.dirichlet([0.3] * 4, size=L).T).astype(np.int64)
        pfm[0, pfm.sum(axis=0) == 0] = 1
        out.append(oracle.pfm_to_pwm(pfm, BG).tolist())
    return out


def _cutoffs(pwms, text, rng, rate=4e-3):
    """About `rate` of the random windows of `text` pass (oracle offset-0 scores of random samples)."""
    lmax = max(len(p[0]) for p in pwms)
    starts = rng.integers(0, len(text) - lmax, 3000)
    samples = [text[a:a + lmax].upper().replace("N", "A") for a in starts.tolist()]
    sc = oracle.score_arrays(pwms, samples, 3)
    k = max(int(len(samples) * rate), 1)
    return [float(np.sort(row)[::-1][k]) for row in sc]


def _vcf_records(texts, rng):
    """(chrom, POS, ID, REF, ALT-field) records covering the hard cases, plus random SNVs / MNVs."""
    recs = []
    acgt = "ACGT"

    def ref_of(c, p, r):
        return texts[c][p:p + r]

    def other(b):
        return acgt[(acgt.find(b.upper()) + 1 + int(rng.integers(3))) % 4] if b.upper() in acgt else acgt[int(rng.integers(4))]

    n1 = len(texts["chr1"])
    for c, p, r in [("chr1", 0, 1), ("chr1", n1 - 1, 1), ("chr1", n1 - 3, 3), ("chr2", 0, 2), ("chrS", 0, 1),
                    ("chrS", len(texts["chrS"]) - 2, 2)]:
        ref = ref_of(c, p, r)
        recs.append((c, p + 1, f"edge{len(recs)}", ref, "".join(other(b) for b in ref)))
    for p in (500, 501, 502):                                    # adjacent variants
        ref = ref_of("chr1", p, 1)
        recs.append(("chr1", p + 1, f"adj{p}", ref, other(ref)))
    ref = ref_of("chr1", 777, 1)                                  # several alleles at one position (one record + one more)
    recs.append(("chr1", 778, "multi", ref, ",".join(b for b in acgt if b != ref.upper())))
    recs.append(("chr1", 778, "multi2", ref, other(ref)))
    ref = ref_of("chr1", 1998, 4)                                 # MNV across the N run's left edge
    recs.append(("chr1", 1999, "acrossN", ref, "GATC"))
    recs.append(("chr1", 2100, "overN", ref_of("chr1", 2099, 1), "C"))   # REF over N
    for p in (1100, 3200, 6000):                                  # ALT == REF (repeat, soft-masked, plain)
        ref = ref_of("chr1", p, 2)
        recs.append(("chr1", p + 1, f"same{p}", ref, ref.upper()))
    recs.append(("chr1", 1201, "repeat", ref_of("chr1", 1200, 1), "G"))  # inside the tandem repeat
    for k in range(120):
        c = "chr1" if k % 3 else "chr2"
        r = 1 if k % 5 else int(rng.integers(2, 4))
        p = int(rng.integers(0, len(texts[c]) - r))
        ref = ref_of(c, p, r)
        recs.append((c, p + 1, f"r{k}", ref, "".join(other(b) for b in ref)))
    recs.append(("chrZ", 5, "unk", "A", "G"))                     # skipped records ride along
    recs.append(("chr1", 10, "ind", ref_of("chr1", 9, 1), "AT"))
    return recs


def _write_vcf(path, recs):
    with open(path, "w") as fh:
        fh.write(VCF_HEADER + "".join(f"{c}\t{p}\t{i}\t{r}\t{a}\t.\tPASS\t.\n" for c, p, i, r, a in recs))


@pytest.fixture(scope="module")
def setup(tmp_path_factory):
    rng = np.random.default_rng(23)
    texts = {}
    for name, n in [("chr1", 9000), ("chr2", 3000), ("chrS", 20)]:
        s = bytearray(synth.random_bases(rng, n).tobytes())
        if n == 9000:
            s[1000:1400] = b"AT" * 200                            # tandem repeat
            s[2000:2300] = b"N" * 300                             # N run
            s[3000:3500] = bytes(s[3000:3500]).lower()            # soft-masked
            s[4000:4003] = b"RYN"                                 # IUPAC codes
        texts[name] = bytes(s).decode()
    chroms = sorted(texts)
    packs = [synth.pack_ascii(np.frombuffer(texts[c].encode(), dtype=np.uint8)) for c in chroms]
    pg = PackedGenome(chroms, {c: len(texts[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                      np.concatenate([p[1] for p in packs]), name="vg")
    pwms = _pwms(rng, 22, 6, 30) + _pwms(rng, 4, 33, 40) + _pwms(rng, 2, 65, 70)
    cutoffs = _cutoffs(pwms, texts["chr1"][4100:] + texts["chr2"], rng)
    cutoffs[3] = 0.0                                              # every all-N window and many others pass
    recs = _vcf_records(texts, rng)
    root = tmp_path_factory.mktemp("variants")
    vcf = root / "calls.vcf"
    _write_vcf(vcf, recs)
    variants = read_vcf(str(vcf), pg)
    # cutoffs exactly on window scores: motif 5 on a ref window, motif 24 (33-40 columns) on an alt window
    for m, a, use_alt in ((5, 7, False), (24, 12, True)):
        L = len(pwms[m][0])
        c, p = variants.chroms[variants.chrom[a]], int(variants.pos[a])
        s = max(p - L + 1, 0)
        win = texts[c][s:s + L]
        if use_alt:
            k = p - s
            win = win[:k] + variants.alt[a] + win[k + len(variants.alt[a]):]
        cutoffs[m] = float(oracle.score_arrays([pwms[m]], [win], 1)[0, 0])
    return dict(texts=texts, pg=pg, pwms=pwms, cutoffs=cutoffs, variants=variants, recs=recs, root=root)


def oracle_rows(setup, strand, pwms=None, cutoffs=None):
    """Rows (allele, motif, chromosome start, strand, ref_score, alt_score, effect) in the contract's order."""
    texts, v = setup["texts"], setup["variants"]
    pwms = pwms or setup["pwms"]
    cutoffs = cutoffs if cutoffs is not None else setup["cutoffs"]
    lens = [len(p[0]) for p in pwms]
    lmax = max(lens)
    seqs, meta = [], []
    for a in range(len(v)):
        c, p, alt = v.chroms[v.chrom[a]], int(v.pos[a]), v.alt[a]
        r = len(alt)
        cs, ce = max(p - lmax + 1, 0), min(p + r + lmax - 1, len(texts[c]))
        ref_ctx = texts[c][cs:ce]
        alt_ctx = ref_ctx[:p - cs] + alt + ref_ctx[p - cs + r:]
        seqs += [ref_ctx, alt_ctx]
        meta.append((cs, p - cs, r))
    counts, seq_idx, start, score, strd = oracle.scan_arrays(pwms, cutoffs, seqs, STRAND[strand], n_threads=8)
    motif_of = np.repeat(np.arange(len(pwms)), counts)
    hits = {}
    for m, q, s, sc, x in zip(motif_of.tolist(), seq_idx.tolist(), start.tolist(), score.tolist(), strd.tolist()):
        a, side = divmod(q, 2)
        cs, c0, r = meta[a]
        if s + lens[m] <= c0 or s >= c0 + r:
            continue
        hits.setdefault((a, m, s, x), [None, None])[side] = sc
    # the missing side, scored by the oracle's c_score on the L-base window
    todo = {}
    for key, sides in hits.items():
        for side in (0, 1):
            if sides[side] is None:
                a, m, s, x = key
                todo.setdefault((m, x), []).append((key, side, seqs[2 * a + side][s:s + lens[m]]))
    for (m, x), items in todo.items():
        sc = oracle.score_arrays([pwms[m]], [w for _, _, w in items], x)[0]
        for (key, side, _), val in zip(items, sc.tolist()):
            hits[key][side] = val
    rows = []
    for (a, m, s, x), (rs, al) in sorted(hits.items()):
        ref_hit, alt_hit = rs - cutoffs[m] >= -1e-10, al - cutoffs[m] >= -1e-10
        assert ref_hit or alt_hit
        rows.append((a, m, meta[a][0] + s, x, rs, al, 3 if ref_hit and alt_hit else (1 if ref_hit else 2)))
    return rows


def assert_rows(sites, rows):
    cols = list(zip(*rows)) if rows else [[]] * 7
    assert len(sites) == len(rows)
    assert np.array_equal(sites.allele, np.array(cols[0], np.int32))
    assert np.array_equal(sites.motif, np.array(cols[1], np.int32))
    assert np.array_equal(sites.start, np.array(cols[2], np.int64))
    assert np.array_equal(sites.strand, np.array(cols[3], np.int8))
    assert np.array_equal(sites.ref_score.view(np.uint64), np.array(cols[4], np.float64).view(np.uint64))
    assert np.array_equal(sites.alt_score.view(np.uint64), np.array(cols[5], np.float64).view(np.uint64))
    assert np.array_equal(sites.effect, np.array(cols[6], np.int8))


def test_extract_subst_equals_host_encoding(setup):
    texts, v, pg = setup["texts"], setup["variants"], setup["pg"]
    ctx = engine.Context(0)
    dg = DeviceGenome(pg, ctx=ctx)
    try:
        idx = np.array([dg.chrom_index[v.chroms[c]] for c in v.chrom], dtype=np.int32)
        cs = np.maximum(v.pos - 37, 0)
        ce = np.minimum(v.pos + 41, np.array([pg.chrom_sizes[v.chroms[c]] for c in v.chrom]))
        r = np.array([len(x) for x in v.alt])
        sub_off = np.concatenate([[0], np.cumsum(r)])
        sub_pos = np.concatenate([np.arange(k) + (p - a) for k, p, a in zip(r, v.pos, cs)])
        sub_code = np.array(["ACGT".index(b) for b in "".join(v.alt).upper()], dtype=np.uint8)
        alt = dg.seqs.extract_subst(idx, cs, ce, sub_off, sub_pos, sub_code)
        want = []
        for a in range(len(v)):
            c, p = v.chroms[v.chrom[a]], int(v.pos[a])
            t = texts[c][cs[a]:ce[a]]
            want.append(t[:p - cs[a]] + v.alt[a] + t[p - cs[a] + r[a]:])
        assert np.array_equal(alt.codes(), np.concatenate([oracle.encode(w) for w in want]))
        alt.close()
        empty = dg.seqs.extract_subst(idx[:0], cs[:0], ce[:0], [0], [], [])
        assert empty.n == 0
        empty.close()
        with pytest.raises(ValueError):
            dg.seqs.extract_subst(idx[:1], cs[:1], ce[:1], [0, 1], [int(ce[0] - cs[0])], [0])   # outside the sequence
    finally:
        dg.close()
        ctx.close()


@pytest.mark.parametrize("strand", ["+", "-", "both"])
def test_rows_equal_oracle(setup, strand):
    rows = oracle_rows(setup, strand)
    sites = scan_variants(setup["pg"], setup["pwms"], setup["cutoffs"], setup["variants"], strand=strand)
    assert_rows(sites, rows)
    if strand == "both":
        by = sites.rows_by_effect()
        assert by["gain"] > 0 and by["loss"] > 0 and by["both"] > 0
        cut = setup["cutoffs"]
        for m in (5, 24):                                         # the exact-cutoff windows are rows
            assert any(r[1] == m and (r[4] == cut[m] or r[5] == cut[m]) for r in rows)
        assert any(r[1] >= 26 for r in rows)                      # the > 64-column route produced rows
        v = setup["variants"]
        same = {a for a in range(len(v)) if v.alt[a].upper() == v.ref[a].upper()}
        sel = np.isin(sites.allele, list(same))
        assert sel.sum() > 0 and (sites.effect[sel] == 3).all()
        assert np.array_equal(sites.ref_score[sel].view(np.uint64), sites.alt_score[sel].view(np.uint64))
        assert v.skipped["unknown_chrom"] == 1 and v.skipped["unsupported"] == 1


def test_overflow_retry_keeps_rows(setup):
    rows = oracle_rows(setup, "both")
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


def test_cli_tables_equal_oracle(setup, tmp_path):
    gdir, mdir = tmp_path / "vg", tmp_path / "vm"
    gdir.mkdir(), mdir.mkdir()
    with open(gdir / "vg.fa", "w") as fh:
        for c in sorted(setup["texts"]):
            t = setup["texts"][c]
            fh.write(f">{c}\n" + "".join(t[i:i + 60] + "\n" for i in range(0, len(t), 60)))
    pw = MotifPwms(name="vm", genome="vg")
    for k, (m, c) in enumerate(zip(setup["pwms"], setup["cutoffs"])):
        pw.append(PositionWeightMatrix(np.array(m), name=f"TF{k}", matrix_id=f"MA{k:04d}.1", cutoffs={"1e-4": c}))
    pw.write_motifscan_pwms(str(mdir / "vm_vg_pwms.motifscan"))
    back = MotifPwms()
    back.read_motifscan_pwms(str(mdir / "vm_vg_pwms.motifscan"))
    pwms, cutoffs = [p.matrix for p in back], [p.cutoffs["1e-4"] for p in back]
    vcf = tmp_path / "calls.vcf"
    _write_vcf(vcf, setup["recs"])
    out = tmp_path / "out"
    assert cli.main(["variant", "-i", str(vcf), "-m", str(mdir), "-g", str(gdir), "-o", str(out), "-t", "4"]) == 0
    v = setup["variants"]
    rows = oracle_rows(setup, "both", pwms=pwms, cutoffs=cutoffs)
    names = {1: "loss", 2: "gain", 3: "both"}
    want = msio.VARIANT_SITES_HEADER + "".join(
        f"{v.chroms[v.chrom[a]]}\t{v.pos[a] + 1}\t{v.id[a]}\t{v.ref[a]}\t{v.alt[a]}\t{back[m].matrix_id}\t{back[m].name}\t"
        f"{s}\t{s + back[m].length}\t{'+' if x == 1 else '-'}\t{rs}\t{al}\t{names[e]}\n" for a, m, s, x, rs, al, e in rows)
    assert (out / "motif_variant_sites.xls").read_text() == want
    summ = msio.VARIANT_SUMMARY_HEADER
    for m, p in enumerate(back):
        n = [len({r[0] for r in rows if r[1] == m and r[6] == e}) for e in (2, 1, 3)]
        summ += f"{p.matrix_id}\t{p.name}\t{n[0]}\t{n[1]}\t{n[2]}\n"
    assert (out / "motif_variant_summary.xls").read_text() == summ
    # an empty VCF: the sites table is its header; the summary lists every motif with zero counts
    empty = tmp_path / "empty.vcf"
    empty.write_text(VCF_HEADER)
    out2 = tmp_path / "out2"
    assert cli.main(["variant", "-i", str(empty), "-m", str(mdir), "-g", str(gdir), "-o", str(out2)]) == 0
    assert (out2 / "motif_variant_sites.xls").read_text() == msio.VARIANT_SITES_HEADER
    assert (out2 / "motif_variant_summary.xls").read_text() == msio.VARIANT_SUMMARY_HEADER + "".join(
        f"{p.matrix_id}\t{p.name}\t0\t0\t0\n" for p in back)
    for bad in (["-i", str(tmp_path / "missing.vcf")], ["-i", str(vcf), "-p", "1e-6"]):
        with pytest.raises(SystemExit):
            cli.main(["variant", "-m", str(mdir), "-g", str(gdir), "-o", str(tmp_path / "x")] + bad)
