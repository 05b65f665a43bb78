"""`motifscan variant --haplotypes` host side: genotype parsing in read_vcf(samples=...) with every GT form and skip
reason, its errors, the clustering of each haplotype's alleles (haplotype_clusters: gap rule, chains, chromosome
boundaries, conflicts, de-duplication, indel trimming) and the native haplotype-table writer against Python's str().
No GPU."""
import numpy as np
import pytest

from motifscan_b200 import io as msio
from motifscan_b200 import synth
from motifscan_b200.genome import PackedGenome
from motifscan_b200.variants import (CALL_SKIP_REASONS, SKIP_REASONS, HaplotypeSites, Variants, haplotype_clusters,
                                     read_vcf)

TEXTS = {"chrA": b"ACGTNNacgtACGTRYACGTTTGCAacgtNNNN", "chrB": b"GATTACAGATTACA"}
HEADER = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\tS3\n"


def _packed():
    chroms = sorted(TEXTS)
    packs = [synth.pack_ascii(np.frombuffer(TEXTS[c], dtype=np.uint8)) for c in chroms]
    return PackedGenome(chroms, {c: len(TEXTS[c]) for c in chroms}, np.concatenate([p[0] for p in packs]),
                        np.concatenate([p[1] for p in packs]))


def _write(path, records, header=HEADER):
    path.write_text(header + "".join("\t".join(map(str, r)) + "\n" for r in records))


RECORDS = [  # chrom, POS, ID, REF, ALT, QUAL, FILTER, INFO, FORMAT, S1, S2, S3
    ("chrB", 2, "snv", "A", "C", ".", "PASS", ".", "GT", "0|1", "1|0:7", "1/1"),
    ("chrB", 4, "multi", "T", "C,<INS>", ".", "PASS", ".", "GT:DP", "1|2:5", "2/2:3", "0/1"),
    ("chrB", 6, "miss", "C", "G", ".", "PASS", ".", "GT", "./.", ".|1", "1"),
    ("chrB", 8, "nogt", "G", "T", ".", "PASS", ".", "DP:GT", "3:1|1", "4:1|1", "5:0|1"),
    ("chrB", 9, "mism", "C", "A", ".", "PASS", ".", "GT", "1|1", "0|0", "0"),      # genome T: ref_mismatch
    ("chrB", 10, "het2", "T", "A,G", ".", "PASS", ".", "GT", "1/2", "2|1", "0/2"),
    ("chrZ", 1, "unk", "A", "T", ".", "PASS", ".", "GT", "1|1", "0|0", "0|0"),
]


def test_read_vcf_genotypes_and_call_skips(tmp_path):
    pg = _packed()
    path = tmp_path / "calls.vcf"
    _write(path, RECORDS)
    v = read_vcf(str(path), pg, samples="all")
    assert v.samples == ["S1", "S2", "S3"]
    assert v.id == ["snv", "multi", "miss", "nogt", "het2", "het2"]
    assert v.skipped == {"unknown_chrom": 1, "out_of_range": 0, "unsupported": 1, "ref_mismatch": 1}
    got = sorted(zip(np.array(v.id)[v.call_allele].tolist(), [v.alt[a] for a in v.call_allele],
                     v.call_sample.tolist(), v.call_hap.tolist()))
    want = sorted([("snv", "C", 0, 1), ("snv", "C", 1, 0), ("snv", "C", 2, 0), ("snv", "C", 2, 1),
                   ("multi", "C", 0, 0),
                   ("miss", "G", 1, 1), ("miss", "G", 2, 0),
                   ("het2", "G", 1, 0), ("het2", "A", 1, 1)])
    assert got == want
    # missing: ./. (2) + .|1 (1) + three samples without GT; unphased: 0/1, 1/2 (2), 0/2;
    # allele_skipped: 1|2 -> <INS>, 2/2 -> <INS> twice, 1|1 of the ref_mismatch allele, 1|1 of the unknown chrom (twice)
    assert v.call_skipped == {"missing": 6, "unphased": 4, "allele_skipped": 7}
    # a list reads only those samples, in its order
    w = read_vcf(str(path), pg, samples=["S3", "S1"])
    assert w.samples == ["S3", "S1"]
    assert sorted(zip(w.call_allele.tolist(), w.call_sample.tolist(), w.call_hap.tolist())) == sorted(
        [(0, 0, 0), (0, 0, 1), (0, 1, 1), (1, 1, 0), (2, 0, 0)])
    assert w.call_skipped == {"missing": 4, "unphased": 4, "allele_skipped": 5}
    # the default ignores the sample columns and reads the same alleles
    d = read_vcf(str(path), pg)
    assert d.samples == [] and len(d.call_allele) == 0 and d.call_skipped == dict.fromkeys(CALL_SKIP_REASONS, 0)
    assert (d.id, d.alt, d.skipped) == (v.id, v.alt, v.skipped)
    with pytest.raises(ValueError, match="S9"):
        read_vcf(str(path), pg, samples=["S1", "S9"])


def test_read_vcf_without_samples_is_an_error_with_samples(tmp_path):
    pg = _packed()
    path = tmp_path / "plain.vcf"
    _write(path, [r[:8] for r in RECORDS], header="##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
    assert len(read_vcf(str(path), pg)) == 6
    with pytest.raises(ValueError, match="no sample columns"):
        read_vcf(str(path), pg, samples="all")


@pytest.mark.parametrize("gt, what", [("0|1|1", "ploidy 3"), ("0/3", "GT allele 3"), ("x|1", "'x' is not an integer"),
                                      ("1|-1", "GT allele -1")])
def test_read_vcf_bad_genotypes_name_their_line(tmp_path, gt, what):
    pg = _packed()
    path = tmp_path / "bad.vcf"
    recs = [RECORDS[0], ("chrB", 10, "het2", "T", "A,G", ".", "PASS", ".", "GT", "0|0", gt, "0|0")]
    _write(path, recs)
    with pytest.raises(ValueError, match=f"line 4: .*{what}"):
        read_vcf(str(path), pg, samples="all")
    assert len(read_vcf(str(path), pg)) == 3                  # without genotypes the line is fine


def _variants(alleles, calls, indels=False, samples=("S1", "S2")):
    """Variants from (chrom index, 0-based pos, REF, ALT, ID) and (allele, sample, hap) calls."""
    c, p, r, a, i = zip(*alleles)
    ca, cs, ch = zip(*calls) if calls else ((), (), ())
    return Variants(["chrA", "chrB"], c, p, r, a, i, range(len(c)), dict.fromkeys(SKIP_REASONS, 0), len(c),
                    indels=indels, samples=samples, call_allele=ca, call_sample=cs, call_hap=ch)


def _clusters(h):
    return [tuple(h.allele[h.allele_off[k]:h.allele_off[k + 1]].tolist()) for k in range(len(h))]


def _carriers(h):
    return [list(zip(h.carrier_sample[h.carrier_off[k]:h.carrier_off[k + 1]].tolist(),
                     h.carrier_hap[h.carrier_off[k]:h.carrier_off[k + 1]].tolist())) for k in range(len(h))]


def test_clusters_gap_chain_and_chromosome_boundaries():
    alleles = [(0, 10, "A", "C", "a"), (0, 19, "A", "C", "b"), (0, 20, "A", "C", "c"), (0, 40, "AC", "GT", "d"),
               (0, 49, "A", "T", "e"), (0, 55, "A", "T", "f"), (1, 9, "A", "T", "g"), (1, 12, "A", "T", "h")]
    lmax = 10                                     # joined when p2 - (p1 + r1) <= 8
    calls = [(0, 0, 0), (1, 0, 0),                # 10 and 19: gap 8, joined
             (0, 0, 1), (2, 0, 1),                # 10 and 20: gap 9, split
             (3, 1, 0), (4, 1, 0), (5, 1, 0),     # MNV [40, 42), 49 (gap 7), 55 (gap 5): a chain of three
             (5, 1, 1), (6, 1, 1), (7, 1, 1)]     # chrA 55 and chrB 9 never join; chrB 9 and 12 do
    h = haplotype_clusters(_variants(alleles, calls), lmax)
    assert _clusters(h) == [(0,), (0, 1), (2,), (3, 4, 5), (5,), (6, 7)]
    assert h.chrom.tolist() == [0, 0, 0, 0, 0, 1]
    assert _carriers(h) == [[(0, 1)], [(0, 0)], [(0, 1)], [(1, 0)], [(1, 1)], [(1, 1)]]
    assert h.overlap == 0 and h.sizes().tolist() == [1, 2, 1, 3, 1, 2]


def test_clusters_conflicts_and_deduplication():
    alleles = [(0, 10, "A", "ATT", "i1"), (0, 10, "A", "AG", "i2"),        # two insertions at one point
               (0, 20, "ACGT", "A", "del"), (0, 22, "G", "C", "in_del"),    # an SNV inside a deletion
               (0, 30, "A", "C", "s1"), (0, 31, "C", "G", "s2"), (0, 25, "T", "A", "s0")]
    calls = [(0, 0, 0), (1, 0, 0),                # i2 conflicts with i1 (the smaller allele index first at a tie)
             (2, 0, 1), (3, 0, 1), (4, 0, 1),     # in_del dropped; s1 then compared with the deletion, kept
             (4, 1, 0), (5, 1, 0), (4, 1, 1), (5, 1, 1), (4, 0, 0), (5, 0, 0),
             (6, 1, 0)]
    h = haplotype_clusters(_variants(alleles, calls, indels=True), 12)
    assert h.overlap == 2
    # S1 h0: i1 [10] ... s1 s2 (gap 30 - 11 = 19 > 10: apart); S1 h1: del [21, 24) + s1 (gap 6) one cluster;
    # S2 h0: s0 (25), s1 (gap 4), s2: one cluster; s1 s2 are carried by S1 h0 and S2 h1
    assert _clusters(h) == [(0,), (2, 4), (6, 4, 5), (4, 5)]
    assert _carriers(h) == [[(0, 0)], [(0, 1)], [(1, 0)], [(0, 0), (1, 1)]]


def test_clusters_use_the_trimmed_change_in_indel_mode():
    # a deletion with its anchor base at 10 removes [11, 13): an SNV at 1 is 9 bases from the trimmed change (split at
    # lmax 10) but 8 from the untrimmed one; one at 21 is 8 bases behind it (joined); an SNV on the anchor (S2) does
    # not conflict with it
    alleles = [(0, 10, "GAT", "G", "del"), (0, 10, "G", "C", "anchor"), (0, 1, "C", "A", "left"), (0, 21, "A", "C", "right")]
    calls = [(0, 0, 0), (2, 0, 0), (3, 0, 0), (0, 1, 0), (1, 1, 0)]
    h = haplotype_clusters(_variants(alleles, calls, indels=True), 10)
    assert h.overlap == 0
    assert _clusters(h) == [(2,), (1, 0), (0, 3)]
    assert h.p.tolist()[:2] == [11, 10] and h.r.tolist()[:2] == [2, 1]


class _Pwm:
    def __init__(self, matrix_id, name, length):
        self.matrix_id, self.name, self.length = matrix_id, name, length


def test_native_haplotype_writer_against_str(tmp_path):
    alleles = [(0, 10, "A", "C", "rs1"), (0, 12, "AT", "A", "rs2"), (1, 3, "G", "T", ".")]
    calls = [(0, 0, 0), (1, 0, 0), (0, 1, 1), (1, 1, 1), (2, 1, 0)]
    v = _variants(alleles, calls, indels=True)
    h = haplotype_clusters(v, 8)
    assert _clusters(h) == [(0, 1), (2,)]
    pwms = [_Pwm("MA0001.1", "TF-a", 7), _Pwm("MA0002.1", "TF:b", 12)]
    nan = float("nan")
    rows = [  # cluster, motif, strand, ref_start, alt_start, ref, alt, effect, paired
        (0, 0, 1, 5, 5, 1e-5, 0.1 + 0.2, 3, True),
        (0, 0, 2, 9, -1, -0.0, nan, 1, False),
        (0, 1, 1, -1, 11, nan, 1e16, 2, False),
        (0, 1, 2, 12, 11, 5e-324, nan, 1, True),          # a real NaN score on a paired row is printed as nan
        (1, 1, 2, 0, 0, 1.7976931348623157e308, -7.0, 2, True),
    ]
    cols = list(zip(*rows))
    sites = HaplotypeSites(len(h), 2, *[np.array(c) for c in cols], carrier_off=h.carrier_off,
                           carrier_id=h.carrier_sample.astype(np.int64) * 2 + h.carrier_hap)
    msio.write_haplotype_tables(str(tmp_path), pwms, h, sites)
    names = {1: "loss", 2: "gain", 3: "both"}
    want = msio.HAPLOTYPE_SITES_HEADER
    for c, m, x, rs, at, sr, sa, e, pd in rows:
        ids = "rs1,rs2" if c == 0 else "."
        win = lambda s: "NA\tNA" if s < 0 else f"{s}\t{s + pwms[m].length}"    # noqa: E731
        rtxt = "NA" if not pd and e == 2 else str(float(sr))
        atxt = "NA" if not pd and e == 1 else str(float(sa))
        want += (f"{'chrA' if c == 0 else 'chrB'}\t{c}\t{ids}\t{pwms[m].matrix_id}\t{pwms[m].name}\t{win(rs)}\t"
                 f"{win(at)}\t{'+' if x == 1 else '-'}\t{rtxt}\t{atxt}\t{names[e]}\n")
    assert (tmp_path / "motif_haplotype_sites.xls").read_text() == want
    assert "\tnan\t" in want and "\tNA\t" in want and "NA\tNA" in want
    assert (tmp_path / "motif_haplotype_clusters.xls").read_text() == (
        msio.HAPLOTYPE_CLUSTERS_HEADER + "0\tchrA\t11:A>C,13:AT>A\trs1,rs2\tS1:1,S2:2\n1\tchrB\t4:G>T\t.\tS2:1\n")
    # TF-a: cluster 0 with both and loss rows; TF:b: cluster 0 gain + loss, cluster 1 gain (carried by S2:1)
    assert (tmp_path / "motif_haplotype_summary.xls").read_text() == (
        msio.HAPLOTYPE_SUMMARY_HEADER + "MA0001.1\tTF-a\t0\t1\t1\t0\t2\t2\nMA0002.1\tTF:b\t2\t1\t0\t3\t2\t0\n")
    bad = HaplotypeSites(len(h), 2, [0], [0], [1], [0], [0], [1.0], [1.0], [3], [False])
    with pytest.raises(ValueError, match="effect"):
        msio.write_haplotype_tables(str(tmp_path / "bad"), pwms, h, bad)
    empty = HaplotypeSites(len(h), 2, *[[]] * 9, carrier_off=h.carrier_off)
    msio.write_haplotype_tables(str(tmp_path / "empty"), pwms, h, empty)
    assert (tmp_path / "empty" / "motif_haplotype_sites.xls").read_text() == msio.HAPLOTYPE_SITES_HEADER
