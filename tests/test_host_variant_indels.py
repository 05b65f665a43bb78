"""`motifscan variant --indels` host side: which alleles read_vcf(indels=True) keeps and how it counts the others, the
trimming of REF / ALT to the changed bases, and the native variant-table writer with unpaired rows (effects 5 / 6,
`NA` for the missing score) against Python's str().  No GPU."""
import numpy as np
import pytest

from motifscan_b200 import io as msio
from motifscan_b200 import synth
from motifscan_b200.genome import PackedGenome
from motifscan_b200.variants import SKIP_REASONS, Variants, VariantSites, _trim, read_vcf

TEXTS = {"chrA": b"ACGTNNacgtACGTRYACGTTTGCAacgtNNNN", "chrB": b"GATTACA"}
HEADER = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
RECORDS = [
    ("chrB", 2, "del", "AT", "A"),           # pure deletion of one base
    ("chrB", 2, "ins", "A", "ATTG"),         # pure insertion of three bases
    ("chrA", 1, "cx", "ACG", "TT"),          # complex allele at POS 1
    ("chrA", 1, "ins0", "A", "GA"),          # insertion before the first base (common suffix)
    ("chrB", 7, "insend", "A", "AG"),        # insertion after the last base
    ("chrA", 5, "overN", "NNa", "T"),        # REF over N and a soft-masked base
    ("chrA", 7, "lc", "acg", "a"),           # lower case REF and ALT
    ("chrA", 8, "case", "CGT", "cA"),        # prefix compared ignoring case: "C"/"c" is common
    ("chrB", 2, "star", "A", "*"),           # unsupported
    ("chrB", 2, "dot", "A", "."),            # unsupported
    ("chrB", 2, "sym", "A", "<DEL>"),        # unsupported
    ("chrB", 2, "altn", "A", "AN"),          # N in ALT: unsupported
    ("chrB", 4, "multi", "T", "C,TAA,<INS>"),   # multi-allelic: SNV + insertion + symbolic
    ("chrA", 11, "mm", "GG", "G"),           # genome "AC": ref_mismatch
    ("chrB", 7, "past", "AC", "A"),          # REF runs past the end: out_of_range
    ("chrZ", 1, "unk", "A", "AT"),           # unknown_chrom
    ("chrB", 3, "same", "TT", "TT"),         # equal length, ALT == REF: scanned, not trimmed
    ("chrB", 1, "mnv", "GA", "CC"),          # MNV: scanned as today
]
# scanned alleles: (id, p', r', inserted ALT bases); equal-length alleles keep their full REF / ALT
TRIMMED = {"del": (2, 1, ""), "ins": (2, 0, "TTG"), "cx": (0, 3, "TT"), "ins0": (0, 0, "G"), "insend": (7, 0, "G"),
           "overN": (4, 3, "T"), "lc": (7, 2, ""), "case": (8, 2, "A"), "multi": [(3, 1, "C"), (4, 0, "AA")],
           "same": (2, 2, "TT"), "mnv": (0, 2, "CC")}


def _packed():
    chroms = sorted(TEXTS)
    packs = [synth.pack_ascii(np.frombuffer(TEXTS[c], dtype=np.uint8)) for c in chroms]
    return PackedGenome(chroms, {c: len(TEXTS[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                        np.concatenate([p[1] for p in packs]))


def _write(path, records=RECORDS):
    path.write_text(HEADER + "".join(f"{c}\t{p}\t{i}\t{r}\t{a}\t.\tPASS\t.\n" for c, p, i, r, a in records))


def test_read_vcf_indels_alleles_and_skips(tmp_path):
    pg = _packed()
    path = tmp_path / "calls.vcf"
    _write(path)
    v = read_vcf(str(path), pg, indels=True)
    assert v.indels and v.n_records == len(RECORDS)
    assert v.skipped == {"unknown_chrom": 1, "out_of_range": 1, "unsupported": 5, "ref_mismatch": 1}
    got = [(pg.chroms[c], int(p), i, r, a, int(k)) for c, p, i, r, a, k in zip(v.chrom, v.pos, v.id, v.ref, v.alt, v.record)]
    want = []
    for k, (c, p, i, r, alts) in enumerate(RECORDS):
        for a in alts.split(","):
            if i in TRIMMED and not a.startswith("<"):
                want.append((c, p - 1, i, r, a, k))
    assert got == want
    # the default still counts every indel as unsupported
    d = read_vcf(str(path), pg)
    assert not d.indels
    assert [x for x in d.id] == ["multi", "same", "mnv"]
    assert d.skipped == {"unknown_chrom": 1, "out_of_range": 1, "unsupported": 15, "ref_mismatch": 0}


def test_trim_is_the_change(tmp_path):
    pg = _packed()
    path = tmp_path / "calls.vcf"
    _write(path)
    v = read_vcf(str(path), pg, indels=True)
    p, r, first, a = _trim(v)
    alts = "".join(v.alt)
    got = {}
    for k, i in enumerate(v.id):
        got.setdefault(i, []).append((int(p[k]), int(r[k]), alts[first[k]:first[k] + a[k]]))
    want = {i: (t if isinstance(t, list) else [t]) for i, t in TRIMMED.items()}
    assert got == want
    # the change applied to the reference gives the ALT haplotype
    for k in range(len(v)):
        c = pg.chroms[v.chrom[k]]
        text = TEXTS[c].decode()
        hap = text[:v.pos[k]] + v.alt[k] + text[v.pos[k] + len(v.ref[k]):]
        ins = alts[first[k]:first[k] + a[k]]
        assert (text[:p[k]] + ins + text[p[k] + r[k]:]).upper() == hap.upper()


class _Pwm:
    def __init__(self, matrix_id, name, length):
        self.matrix_id, self.name, self.length = matrix_id, name, length


def test_native_writer_unpaired_rows(tmp_path):
    v = Variants(["chr1"], [0, 0, 0], [10, 20, 30], ["A", "AT", "C"], ["AGG", "A", "T"], ["i1", "d1", "s1"],
                 [0, 1, 2], dict.fromkeys(SKIP_REASONS, 0), 3, indels=True)
    pwms = [_Pwm("MA0001.1", "TF-a", 7), _Pwm("MA0002.1", "TF:b", 12)]
    nan = float("nan")
    rows = [  # allele, motif, start, strand, ref, alt, effect, paired
        (0, 0, 5, 1, nan, 0.1 + 0.2, 2, False),
        (0, 1, 6, 2, 1e-5, 3.0, 3, True),
        (1, 0, 19, 1, -0.0, nan, 1, False),
        (1, 0, 20, 2, 5e-324, nan, 1, False),      # a real NaN score on a paired row is printed as nan
        (1, 1, 21, 1, 1e16, 12.0000001, 2, True),
        (2, 0, 25, 2, 1.7976931348623157e308, -7.0, 1, True),
    ]
    cols = list(zip(*rows))
    sites = VariantSites(3, 2, *[np.array(c) for c in cols[:7]], paired=np.array(cols[7]))
    sites.paired[3] = True
    msio.write_variant_tables(str(tmp_path), pwms, v, sites)
    names = {1: "loss", 2: "gain", 3: "both"}
    want = msio.VARIANT_SITES_HEADER
    for a, m, s, x, rs, al, e, pd in rows:
        pd = pd or s == 20
        rtxt = "NA" if not pd and e == 2 else str(float(rs))
        atxt = "NA" if not pd and e == 1 else str(float(al))
        want += (f"chr1\t{v.pos[a] + 1}\t{v.id[a]}\t{v.ref[a]}\t{v.alt[a]}\t{pwms[m].matrix_id}\t{pwms[m].name}\t{s}\t"
                 f"{s + pwms[m].length}\t{'+' if x == 1 else '-'}\t{rtxt}\t{atxt}\t{names[e]}\n")
    assert (tmp_path / "motif_variant_sites.xls").read_text() == want
    assert "\tnan\t" in want and "\tNA\t" in want
    summ = msio.VARIANT_SUMMARY_HEADER + "MA0001.1\tTF-a\t1\t2\t0\nMA0002.1\tTF:b\t1\t0\t1\n"
    assert (tmp_path / "motif_variant_summary.xls").read_text() == summ
    # effects 0 and 4, and 7 (both, unpaired), are not rows
    for eff, paired in ((0, True), (4, True), (3, False)):
        bad = VariantSites(3, 2, [0], [0], [5], [1], [1.0], [1.0], [eff], paired=[paired])
        with pytest.raises(ValueError, match="effect"):
            msio.write_variant_tables(str(tmp_path / f"bad{eff}"), pwms, v, bad)
