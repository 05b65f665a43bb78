"""The native BED writer (msb_write_sites_bed) and cell-table formatter (msb_format_cell_tables) print exactly
what the Python writers print -- `str()` of ints and floats -- on awkward doubles.  Host code only: no GPU."""
import numpy as np

from motifscan_b200 import io as msio
from motifscan_b200.region import GenomicRegion
from motifscan_b200.scanner import MotifSite, MotifSites


class _Pwm:
    def __init__(self, matrix_id, name, length):
        self.matrix_id, self.name, self.length = matrix_id, name, length


AWKWARD = [0.1 + 0.2, 1e-5, -0.0, 1e16, 5e-324, 3.0, -7.0, 123456789.0, 1e22, -2.5e-7, 0.5, 1.7976931348623157e308,
           -1e-4, 12.0000001, 1e15, 9.999999999999999e15]


class _Res:
    """The arrays of a de-duplicated scan result, shaped like what MotifSites reads."""

    def __init__(self, counts, seq_idx, start, score, strand):
        self.offsets = np.zeros(len(counts) + 1, dtype=np.int64)
        np.cumsum(counts, out=self.offsets[1:])
        self.seq_idx, self.start, self.score, self.strand = seq_idx, start, score, strand


def test_native_bed_equals_python_writer(tmp_path):
    from motifscan_b200 import build
    build.build()
    rng = np.random.default_rng(3)
    regions = [GenomicRegion("chr1", 100, 900), GenomicRegion("chr2", 0, 5000), GenomicRegion("chrUn_gl000220", 40, 41)]
    pwms = [_Pwm("MA0001.1", "TF-a", 7), _Pwm("MA0002.1", "TF:b/c", 12), _Pwm("MA0003.1", "empty", 9)]
    n = len(AWKWARD)
    counts = [n, 5, 0]
    seq_idx = np.concatenate([np.sort(rng.integers(0, 3, n)), np.array([0, 0, 1, 2, 2])]).astype(np.int32)
    start = rng.integers(0, 400, len(seq_idx)).astype(np.int32)
    score = np.array(AWKWARD + [2.0, -0.0, 1e-300, 7.25, 1 / 3], dtype=np.float64)
    strand = rng.integers(1, 3, len(seq_idx)).astype(np.int8)
    sites = MotifSites(_Res(counts, seq_idx, start, score, strand), len(pwms), [r.start for r in regions], [p.length for p in pwms])
    msio.write_sites_bed(str(tmp_path / "native"), pwms, regions, sites)
    nested = [[[MotifSite(*s) for s in cell] for cell in per] for per in sites.tolist()]
    msio.write_sites_bed(str(tmp_path / "python"), pwms, regions, nested)
    for pwm in pwms:
        name = msio.replace_special_char(f"{pwm.matrix_id}_{pwm.name}") + "_sites.bed"
        got = (tmp_path / "native" / "motif_sites" / name).read_bytes()
        assert got == (tmp_path / "python" / "motif_sites" / name).read_bytes(), name
    first = (tmp_path / "native" / "motif_sites" / "MA0001_1_TF_a_sites.bed").read_text().splitlines()
    assert sorted(line.split("\t")[4] for line in first) == sorted(str(v) for v in AWKWARD)


def test_cell_tables_equal_python_tables(tmp_path):
    from motifscan_b200 import build
    build.build()
    regions = [GenomicRegion("chr1", 0, 249250621), GenomicRegion("chr2", 0, 243199373), GenomicRegion("chrM", 0, 16571)]
    pwms = [_Pwm(f"MA{k:04d}.1", f"TF{k}", 8) for k in range(len(AWKWARD))]
    rng = np.random.default_rng(4)
    counts = rng.integers(0, 3, (len(regions), len(pwms))).astype(np.int64)
    counts[0, 0] = 3_000_000_000                    # more than an int32 holds
    best = np.array([AWKWARD] * len(regions), dtype=np.float64)
    msio.write_cell_tables(str(tmp_path / "native"), pwms, regions, counts, best)
    header = "chr\tstart\tend\t" + "\t".join(f"{p.matrix_id},{p.name}" for p in pwms) + "\n"
    num, sc = header, header
    for r, g in enumerate(regions):
        lead = f"{g.chrom}\t{g.start + 1}\t{g.end}\t"
        num += lead + "\t".join(str(int(c)) for c in counts[r]) + "\n"
        sc += lead + "\t".join("NA" if c == 0 else str(float(v)) for c, v in zip(counts[r], best[r])) + "\n"
    assert (tmp_path / "native" / "motif_sites_number.xls").read_text() == num
    assert (tmp_path / "native" / "motif_sites_score.xls").read_text() == sc
