"""`motifscan variant` host side: VCF parsing (alleles, skip reasons, gzip, malformed lines) and the native
variant-table writer against Python's str() formatting.  No GPU."""
import gzip

import numpy as np
import pytest

from motifscan_b200 import io as msio
from motifscan_b200 import synth
from motifscan_b200.genome import Genome, PackedGenome
from motifscan_b200.variants import SKIP_REASONS, Variants, VariantSites, read_vcf

TEXTS = {"chrA": b"ACGTNNacgtACGTRYACGTTTGCAacgtNNNN", "chrB": b"GATTACA"}

HEADER = "##fileformat=VCFv4.2\n##contig=<ID=chrA>\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
RECORDS = [
    ("chrA", 1, "rs1", "A", "G"),            # SNV at base 0
    ("chrA", 2, ".", "CG", "TT"),            # MNV
    ("chrA", 4, "m1", "T", "A,C,<DEL>"),     # multi-allelic: two SNVs + a symbolic allele
    ("chrA", 5, "n1", "N", "A"),             # REF over N
    ("chrA", 6, "n2", "NA", "GC"),           # MNV across an N and a soft-masked base, REF in mixed case below
    ("chrA", 7, "lc", "A", "T"),             # genome 'a', REF 'A': case-insensitive match
    ("chrA", 8, "lc2", "cg", "aa"),          # lower-case REF and ALT over lower-case genome
    ("chrA", 15, "iu", "N", "C"),            # genome 'R' (IUPAC), REF 'N': both non-ACGT
    ("chrA", 11, "mm", "C", "T"),            # genome 'A': ref_mismatch
    ("chrA", 16, "iu2", "Y", "A"),           # genome 'Y', REF 'Y': non-ACGT on both sides
    ("chrA", 33, "last", "N", "G"),          # the last base
    ("chrA", 34, "past", "A", "G"),          # behind the end: out_of_range
    ("chrA", 33, "over", "NN", "GG"),        # REF runs past the end: out_of_range
    ("chrA", 0, "zero", "A", "G"),           # POS 0: out_of_range
    ("chrZ", 5, "unk", "A", "G"),            # unknown_chrom
    ("chrB", 2, "ind", "A", "AT"),           # indel: unsupported
    ("chrB", 2, "star", "A", "*"),           # unsupported
    ("chrB", 2, "dot", "A", "."),            # unsupported
    ("chrB", 2, "altn", "A", "N"),           # non-ACGT ALT: unsupported
    ("chrB", 2, "same", "A", "A"),           # ALT == REF: scanned
    ("chrB", 7, "end", "A", "C"),            # last base of chrB
]


def _packed():
    chroms = sorted(TEXTS)
    packs = [synth.pack_ascii(np.frombuffer(TEXTS[c], dtype=np.uint8)) for c in chroms]
    return PackedGenome(chroms, {c: len(TEXTS[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                        np.concatenate([p[1] for p in packs]))


def _vcf_text(records=RECORDS):
    body = "".join(f"{c}\t{p}\t{i}\t{r}\t{a}\t50\tPASS\tDP=3\tGT\t0/1\n" for c, p, i, r, a in records)
    return HEADER + body.replace("n2\tNA", "n2\tNa")


def _expected():
    rows, skipped = [], dict.fromkeys(SKIP_REASONS, 0)
    for rec, (c, p, i, r, alts) in enumerate(RECORDS):
        for a in alts.split(","):
            if c not in TEXTS:
                skipped["unknown_chrom"] += 1
            elif p < 1 or p - 1 + len(r) > len(TEXTS[c]):
                skipped["out_of_range"] += 1
            elif len(a) != len(r) or not set(a) <= set("ACGTacgt"):
                skipped["unsupported"] += 1
            elif i == "mm":
                skipped["ref_mismatch"] += 1
            else:
                rows.append((c, p - 1, i, "Na" if i == "n2" else r, a, rec))
    return rows, skipped


def _check(v, genome_chroms):
    rows, skipped = _expected()
    assert v.skipped == skipped
    assert v.n_records == len(RECORDS)
    got = [(genome_chroms[c], int(p), i, r, a, int(k)) for c, p, i, r, a, k in
           zip(v.chrom, v.pos, v.id, v.ref, v.alt, v.record)]
    assert got == rows


def test_read_vcf_packed_genome(tmp_path):
    pg = _packed()
    path = tmp_path / "calls.vcf"
    path.write_text(_vcf_text())
    v = read_vcf(str(path), pg)
    _check(v, pg.chroms)
    assert len(v) == 13 and v.skipped == {"unknown_chrom": 1, "out_of_range": 3, "unsupported": 5, "ref_mismatch": 1}


def test_read_vcf_gzip_by_magic_and_fasta_genome(tmp_path):
    pg = _packed()
    gz = tmp_path / "calls.txt"                     # no .gz suffix: recognised by its magic bytes
    with gzip.open(gz, "wt") as fh:
        fh.write(_vcf_text())
    _check(read_vcf(str(gz), pg), pg.chroms)
    gdir = tmp_path / "g"
    gdir.mkdir()
    with open(gdir / "g.fa", "wb") as fh:           # the same genome as a FASTA: REF checked on fetched bases
        for c in sorted(TEXTS):
            fh.write(b">" + c.encode() + b"\n" + TEXTS[c][:20] + b"\n" + TEXTS[c][20:] + b"\n")
    genome = Genome("g", path=str(gdir))
    try:
        _check(read_vcf(str(gz), genome), genome.chroms)
    finally:
        genome.close()


def test_read_vcf_empty_and_malformed(tmp_path):
    pg = _packed()
    empty = tmp_path / "empty.vcf"
    empty.write_text(HEADER)
    v = read_vcf(str(empty), pg)
    assert len(v) == 0 and v.n_records == 0 and sum(v.skipped.values()) == 0
    short = tmp_path / "short.vcf"
    short.write_text(HEADER + "chrA\t1\trs1\tA\tG\n" + "chrA\t2\trs2\tC\n")
    with pytest.raises(ValueError, match="line 5"):
        read_vcf(str(short), pg)
    badpos = tmp_path / "badpos.vcf"
    badpos.write_text(HEADER + "\n".join(["chrA\t1\trs1\tA\tG", "chrA\t1\trs1\tA\tG", "chrA\tx2\trs2\tC\tG"]) + "\n")
    with pytest.raises(ValueError, match="line 6"):
        read_vcf(str(badpos), pg)


class _Pwm:
    def __init__(self, matrix_id, name, length):
        self.matrix_id, self.name, self.length = matrix_id, name, length


AWKWARD = [0.1 + 0.2, 1e-5, -0.0, 1e16, 5e-324, 3.0, -7.0, 123456789.0, 1e22, -2.5e-7, 0.5, 1.7976931348623157e308,
           -1e-4, 12.0000001, 1e15, 9.999999999999999e15]


def test_native_variant_table_equals_python_str(tmp_path):
    from motifscan_b200 import build
    build.build()
    rng = np.random.default_rng(11)
    v = Variants(["chr1", "chrUn_gl000220"], [0, 1, 0, 1], [99, 0, 2_000_000_000, 7], ["A", "CG", "t", "N"],
                 ["G", "TT", "a", "C"], ["rs1", ".", "x;y", "id4"], [0, 1, 1, 2], dict.fromkeys(SKIP_REASONS, 0), 3)
    pwms = [_Pwm("MA0001.1", "TF-a", 7), _Pwm("MA0002.1", "TF:b/c", 12), _Pwm("MA0003.1", "never", 9)]
    n = len(AWKWARD)
    allele = np.sort(rng.choice([0, 2, 3], n)).astype(np.int32)          # allele 1 has no row
    motif = rng.integers(0, 2, n).astype(np.int32)
    start = (v.pos[allele] + rng.integers(-6, 2, n)).astype(np.int64)
    strand = rng.integers(1, 3, n).astype(np.int8)
    effect = np.array([1, 2, 3] * 6, dtype=np.int8)[:n]
    ref_score = np.array(AWKWARD, dtype=np.float64)
    alt_score = ref_score[::-1].copy()
    sites = VariantSites(4, 3, allele, motif, start, strand, ref_score, alt_score, effect)
    msio.write_variant_tables(str(tmp_path), pwms, v, sites)
    want = msio.VARIANT_SITES_HEADER
    names = {1: "loss", 2: "gain", 3: "both"}
    for i in range(n):
        a, m = int(allele[i]), int(motif[i])
        want += (f"{v.chroms[v.chrom[a]]}\t{v.pos[a] + 1}\t{v.id[a]}\t{v.ref[a]}\t{v.alt[a]}\t{pwms[m].matrix_id}\t"
                 f"{pwms[m].name}\t{start[i]}\t{start[i] + pwms[m].length}\t{'+' if strand[i] == 1 else '-'}\t"
                 f"{float(ref_score[i])}\t{float(alt_score[i])}\t{names[int(effect[i])]}\n")
    assert (tmp_path / "motif_variant_sites.xls").read_text() == want
    summ = msio.VARIANT_SUMMARY_HEADER
    for m, pwm in enumerate(pwms):
        counts = [len({int(allele[i]) for i in range(n) if motif[i] == m and effect[i] == e}) for e in (2, 1, 3)]
        summ += f"{pwm.matrix_id}\t{pwm.name}\t" + "\t".join(map(str, counts)) + "\n"
    assert (tmp_path / "motif_variant_summary.xls").read_text() == summ
    msio.write_variant_tables(str(tmp_path / "none"), pwms, v, VariantSites(4, 3, *[np.zeros(0)] * 7))
    assert (tmp_path / "none" / "motif_variant_sites.xls").read_text() == msio.VARIANT_SITES_HEADER
    assert (tmp_path / "none" / "motif_variant_summary.xls").read_text() == msio.VARIANT_SUMMARY_HEADER + "".join(
        f"{p.matrix_id}\t{p.name}\t0\t0\t0\n" for p in pwms)
