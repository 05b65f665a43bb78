"""Variant-effect scans: which motif sites do SNVs, MNVs and (opt-in) indels create or destroy (`motifscan variant`).

    variants = read_vcf("calls.vcf.gz", genome)          # alleles + skip counts; indels=True scans indels too
    sites = scan_variants(genome, pwms, cutoffs, variants)
    io.write_variant_tables(out_dir, pwms, variants, sites)

Every ALT of a VCF record is one allele, evaluated alone on the reference background.  An allele is scanned when
its chromosome is in the genome, 1 <= POS and POS - 1 + len(REF) <= the chromosome size, len(ALT) == len(REF) (SNVs
and MNVs), ALT is only A/C/G/T (any case) and REF matches the genome base for base -- the same A/C/G/T ignoring case,
or both not A/C/G/T, which is how scoring sees a base (cscore.c:81-114).  Every other allele is counted under
the first reason it fails, in that order: `unknown_chrom`, `out_of_range`, `unsupported`, `ref_mismatch`.

For an allele at p = POS - 1 with r = len(REF) and a motif of length L the windows are those of the whole-chromosome
scan that overlap the changed bases: starts s with p - L + 1 <= s <= p + r - 1, s >= 0 and s + L <= chromosome size.
A window is a site on an allele when score - cutoff >= -1e-10 (cscore.c:358); a row is a window, strand and motif
that is a site on at least one allele, with its exact score on both and an effect: `loss` (site on ref only),
`gain` (alt only) or `both`.

Indels (read_vcf(indels=True), `motifscan variant --indels`): an allele with len(ALT) != len(REF) is scanned too;
`unsupported` then means only an empty REF, or an ALT that is empty, `.`, `*`, symbolic (`<...>`) or holds a byte
that is not A/C/G/T.  The change is REF and ALT without their longest common prefix and then their longest common
suffix (bases compared under the scoring encoding): r' reference bases at p' replaced by a' inserted ones, r' != a',
one of them possibly 0.  Indels are not left-aligned: one in a repeat is scanned where the VCF puts it, so normalise
the VCF first (e.g. `bcftools norm -f genome.fa`) for positions that do not depend on the caller.  SNVs and MNVs are
not trimmed.  On an allele with changed length k (r' on ref, a' on alt) a window [s, s + L) of the context below
(c = p' relative to it) is affected when s < c + k and s + L > c (for k = 0: it straddles the junction).  It is
paired with the other allele's window at s when s < c + min(r', a') and that window fits in the other context;
paired windows make rows as above.  An unpaired ref site is a `loss` and an unpaired alt site a `gain` whose other
score is missing (NaN, `paired` false; NA in the table).  `start` is the window's position on its allele's haplotype:
left of p' + min(r', a') both haplotypes share coordinates, and only one side ever has unpaired windows.

On the device (msb_scan_variants / msb_scan_variants_ex): each allele's context [max(p - Lmax + 1, 0),
min(p + r + Lmax - 1, size)) (p', r' for an indel) is cut out of the resident genome twice, once as it is and once
with the allele's bases overlaid (msb_seqs_extract_subst) or, in indel mode, spliced in (msb_seqs_extract_splice, every
allele); both context sets go through the ordinary scan pipeline, and a row kernel keeps the sites that touch the
changed bases and scores the same window on the other allele.
"""
import gzip
import logging
import time

import numpy as np

from . import engine

logger = logging.getLogger("motifscan")

SKIP_REASONS = ("unknown_chrom", "out_of_range", "unsupported", "ref_mismatch")
EFFECTS = {1: "loss", 2: "gain", 3: "both"}
STRAND = {"+": 1, "-": 2, "both": 3, 1: 1, 2: 2, 3: 3}

_CODE = np.full(256, 4, dtype=np.uint8)     # A/C/G/T in any case -> 0..3, every other byte -> 4 (cscore.c:91-110)
for _k, _b in enumerate(b"ACGT"):
    _CODE[_b] = _CODE[_b | 0x20] = _k


class Variants:
    """Alleles of a VCF, in input order.  Per allele: `chrom` (index into `chroms`), `pos` (0-based p = POS - 1),
    `ref`, `alt` and `id` as written in the file, and `record` (0-based index of its VCF record among the data lines).
    `skipped`: alleles left out, by reason; `n_records`: data lines read; `indels`: read with indels=True (the
    alleles may change the length, and scan_variants cuts every alt context with a splice)."""

    def __init__(self, chroms, chrom, pos, ref, alt, ids, record, skipped, n_records, indels=False):
        self.indels = bool(indels)
        self.chroms = list(chroms)
        self.chrom = np.asarray(chrom, dtype=np.int32)
        self.pos = np.asarray(pos, dtype=np.int64)
        self.ref, self.alt, self.id = list(ref), list(alt), list(ids)
        self.record = np.asarray(record, dtype=np.int64)
        self.skipped = dict(skipped)
        self.n_records = int(n_records)

    def __len__(self):
        return len(self.pos)


def _open_text(path):
    """A VCF as text lines; gzip (and bgzip) input is recognised by its magic bytes, not by its name."""
    with open(path, "rb") as fh:
        magic = fh.read(2)
    if magic == b"\x1f\x8b":
        return gzip.open(path, "rt", encoding="utf-8", newline=None)
    return open(path, "r", encoding="utf-8", newline=None)


def _genome_planes(genome):
    """(codes, nmask, block_off) of the genome's packed planes in `genome.chroms` order, or None when the genome has
    none (a FASTA-backed `Genome`: its bases are fetched instead)."""
    from .genome import DeviceGenome, PackedGenome
    if isinstance(genome, DeviceGenome):
        if isinstance(genome.genome, PackedGenome):
            genome = genome.genome
        else:
            codes, nmask = genome.seqs.to_packed()
            blocks = np.array([(genome.chrom_sizes[c] + 31) // 32 for c in genome.chroms], dtype=np.int64)
            off = np.zeros(len(blocks) + 1, dtype=np.int64)
            np.cumsum(blocks, out=off[1:])
            return codes, nmask, off
    if isinstance(genome, PackedGenome):
        return genome.codes, genome.nmask, genome.block_off
    return None


def _ref_matches(genome, chrom_idx, pos, refs):
    """Per allele: does REF equal the genome's bases under the scoring encoding?"""
    n = len(refs)
    if n == 0:
        return np.zeros(0, dtype=bool)
    lens = np.fromiter((len(r) for r in refs), dtype=np.int64, count=n)
    want = _CODE[np.frombuffer("".join(refs).encode("latin-1", "replace"), dtype=np.uint8)]
    planes = _genome_planes(genome)
    if planes is None:
        chroms = list(genome.chroms)
        got = np.concatenate([_CODE[np.frombuffer(genome.fetch_bytes(chroms[c], p, p + k) if hasattr(genome, "fetch_bytes")
                                                   else genome.fetch_sequence(chroms[c], p, p + k).encode(), dtype=np.uint8)]
                              for c, p, k in zip(chrom_idx.tolist(), pos.tolist(), lens.tolist())])
    else:
        codes, nmask, block_off = planes
        first = np.zeros(n, dtype=np.int64)
        np.cumsum(lens[:-1], out=first[1:])
        q = np.repeat(pos, lens) + (np.arange(int(lens.sum()), dtype=np.int64) - np.repeat(first, lens))
        b = np.asarray(block_off, dtype=np.int64)[np.repeat(chrom_idx, lens)] + q // 32
        word = np.asarray(codes)[2 * b + (q % 32) // 16]
        got = ((word >> (2 * (q % 16)).astype(np.uint32)) & 3).astype(np.uint8)
        isn = (np.asarray(nmask)[b] >> (q % 32).astype(np.uint32)) & 1
        got[isn == 1] = 4
    same = (got == want).astype(np.int64)
    ends = np.cumsum(lens)
    return np.add.reduceat(same, ends - lens) == lens if n else np.zeros(0, dtype=bool)


def read_vcf(path, genome, indels=False):
    """The alleles of a VCF (see the module docstring for which are scanned) against `genome` (anything with
    `chroms` / `chrom_sizes`; REF is checked against its packed planes when it has them -- `PackedGenome`,
    `DeviceGenome` -- else against its fetched bases).  Lines starting with `#` are skipped; FILTER, INFO and
    sample columns are ignored.  A data line with fewer than 5 tab-separated fields, or a POS that is not an
    integer, raises ValueError naming its line number.  `indels`: also scan alleles whose ALT length differs
    from REF's (else they count as `unsupported`)."""
    chroms = list(genome.chroms)
    index = {c: i for i, c in enumerate(chroms)}
    sizes = [int(genome.chrom_sizes[c]) for c in chroms]
    skipped = dict.fromkeys(SKIP_REASONS, 0)
    chrom, pos, ref, alt, ids, record = [], [], [], [], [], []
    n_records = 0
    acgt = set("ACGTacgt")
    with _open_text(path) as fh:
        for lineno, line in enumerate(fh, 1):
            if line.startswith("#"):
                continue
            line = line.rstrip("\r\n")
            if not line:
                continue
            f = line.split("\t", 5)
            if len(f) < 5:
                raise ValueError(f"{path}: line {lineno}: expected at least 5 tab-separated fields, got {len(f)}")
            try:
                p = int(f[1]) - 1
            except ValueError:
                raise ValueError(f"{path}: line {lineno}: POS {f[1]!r} is not an integer") from None
            rec = n_records
            n_records += 1
            ci = index.get(f[0])
            r = f[3]
            for a in f[4].split(","):
                if ci is None:
                    skipped["unknown_chrom"] += 1
                elif p < 0 or p + len(r) > sizes[ci]:
                    skipped["out_of_range"] += 1
                elif not a or not r or (len(a) != len(r) and not indels) or not acgt.issuperset(a):
                    skipped["unsupported"] += 1
                else:
                    chrom.append(ci)
                    pos.append(p)
                    ref.append(r)
                    alt.append(a)
                    ids.append(f[2])
                    record.append(rec)
    chrom = np.array(chrom, dtype=np.int32)
    pos = np.array(pos, dtype=np.int64)
    ok = _ref_matches(genome, chrom, pos, ref)
    skipped["ref_mismatch"] = int((~ok).sum())
    keep = np.flatnonzero(ok)
    pick = keep.tolist()
    return Variants(chroms, chrom[keep], pos[keep], [ref[i] for i in pick], [alt[i] for i in pick],
                    [ids[i] for i in pick], np.array(record, dtype=np.int64)[keep] if record else np.zeros(0, np.int64),
                    skipped, n_records, indels=indels)


def _trim(variants):
    """Per allele (p', r', first, a'): the change without the longest common prefix and then the longest common suffix
    of REF and ALT (bases compared under the scoring encoding) -- r' bases at p' replaced by the a' bytes from `first`
    on of the concatenated ALTs.  SNVs and MNVs are left as they are."""
    n = len(variants)
    r = np.fromiter((len(x) for x in variants.ref), dtype=np.int64, count=n)
    a = np.fromiter((len(x) for x in variants.alt), dtype=np.int64, count=n)
    rc = _CODE[np.frombuffer("".join(variants.ref).encode("latin-1", "replace"), dtype=np.uint8)]
    ac = _CODE[np.frombuffer("".join(variants.alt).encode("ascii"), dtype=np.uint8)]
    r0, a0 = np.cumsum(r) - r, np.cumsum(a) - a                       # each allele's first byte in rc / ac

    def common(m, ref_at, alt_at):
        """Per allele, the number of leading k < m with rc[ref_at(k)] == ac[alt_at(k)]."""
        who = np.repeat(np.arange(n), m)
        k = np.arange(int(m.sum()), dtype=np.int64) - np.repeat(np.cumsum(m) - m, m)
        out = m.copy()
        diff = rc[ref_at(who, k)] != ac[alt_at(who, k)]
        np.minimum.at(out, who[diff], k[diff])
        return out

    indel = r != a
    m = np.where(indel, np.minimum(r, a), 0)
    pre = common(m, lambda w, k: r0[w] + k, lambda w, k: a0[w] + k)
    m = np.where(indel, np.minimum(r, a) - pre, 0)
    suf = common(m, lambda w, k: r0[w] + r[w] - 1 - k, lambda w, k: a0[w] + a[w] - 1 - k)
    return variants.pos + pre, r - pre - suf, a0 + pre, a - pre - suf


class VariantSites:
    """Rows of a variant scan in (allele, motif, start, strand) order: `allele` (index into the Variants), `motif`
    (index into the motif set), `start` (0-based window start on the chromosome; the window is [start, start + L)),
    `strand` (1 forward, 2 reverse), `ref_score` / `alt_score` (the window's exact score on each allele) and `effect`
    (1 loss, 2 gain, 3 both; `EFFECTS` names them) and `paired` (false for an indel's loss / gain whose window does
    not exist on the other allele: the other score is NaN; a NaN score can also be real, so `paired` is what tells).
    `timings`: device milliseconds per phase; `context_bp`: bases of the ref context set; `motif_bp`: motif x context
    bases scored (both sets); `seconds`: wall time of the scan."""

    def __init__(self, n_alleles, n_motifs, allele, motif, start, strand, ref_score, alt_score, effect, timings=None,
                 context_bp=0, motif_bp=0, seconds=0.0, paired=None):
        self.n_alleles, self.n_motifs = int(n_alleles), int(n_motifs)
        self.allele, self.motif = np.asarray(allele, dtype=np.int32), np.asarray(motif, dtype=np.int32)
        self.start, self.strand = np.asarray(start, dtype=np.int64), np.asarray(strand, dtype=np.int8)
        self.ref_score, self.alt_score = np.asarray(ref_score, dtype=np.float64), np.asarray(alt_score, dtype=np.float64)
        self.effect = np.asarray(effect, dtype=np.int8)
        self.paired = np.ones(len(self.effect), dtype=bool) if paired is None else np.asarray(paired, dtype=bool)
        self.timings = dict(timings or {})
        self.context_bp, self.motif_bp, self.seconds = int(context_bp), int(motif_bp), float(seconds)

    def __len__(self):
        return len(self.allele)

    def rows_by_effect(self):
        return {name: int((self.effect == code).sum()) for code, name in EFFECTS.items()}

    def summary(self):
        """Per motif (set order), the number of alleles with at least one row of each effect:
        dict of int64 arrays n_gain, n_loss, n_both."""
        out = {}
        for code, name in ((2, "n_gain"), (1, "n_loss"), (3, "n_both")):
            sel = self.effect == code
            pairs = np.unique(self.motif[sel].astype(np.int64) * max(self.n_alleles, 1) + self.allele[sel])
            out[name] = np.bincount(pairs // max(self.n_alleles, 1), minlength=self.n_motifs).astype(np.int64)
        return out


def _device_genome(genome, device):
    """(DeviceGenome, owned): the genome resident on `device`, built from its packed planes when it is not already."""
    from .genome import DeviceGenome, PackedGenome
    if isinstance(genome, DeviceGenome):
        return genome, False
    if not isinstance(genome, PackedGenome):
        from . import cli
        genome = cli.packed_genome(genome, cli.PACKED_MIN_BP, device)
    return DeviceGenome(genome, device=device), True


def scan_variants(genome, pwms, cutoffs, variants, strand="both", device=0):
    """Rows of every scanned allele of `variants` (read_vcf) for the motif set `pwms` (4 x L matrices, or objects
    with a `.matrix`) at `cutoffs`, on one GPU.  `genome`: a `DeviceGenome` (used as it is), a `PackedGenome`, or
    a host genome whose packed planes are loaded from (or written to) its cache (`cli.packed_genome`)."""
    mats = [np.asarray(getattr(p, "matrix", p), dtype=np.float64) for p in pwms]
    n, n_motifs = len(variants), len(mats)
    st = STRAND[strand]
    if n == 0 or n_motifs == 0:
        e = np.zeros(0)
        return VariantSites(n, n_motifs, e, e, e, e, e, e, e)
    t0 = time.perf_counter()
    dg, owned = _device_genome(genome, device)
    try:
        ctx = dg.ctx
        lmax = max(m.shape[1] for m in mats)
        cidx = np.array([dg.chrom_index[c] for c in variants.chroms], dtype=np.int32)[variants.chrom]
        size = np.array([dg.chrom_sizes[c] for c in dg.chroms], dtype=np.int64)[cidx]
        if variants.indels:
            p, r, first, a = _trim(variants)
        else:
            p = variants.pos
            r = a = np.fromiter((len(x) for x in variants.ref), dtype=np.int64, count=n)
        cs = np.maximum(p - (lmax - 1), 0)
        ce = np.minimum(p + r + lmax - 1, size)
        core_start = p - cs
        alt_code = _CODE[np.frombuffer("".join(variants.alt).encode("ascii"), dtype=np.uint8)]
        sub_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(a, out=sub_off[1:])
        total = int(sub_off[-1])
        within = np.arange(total, dtype=np.int64) - np.repeat(sub_off[:-1], a)    # k-th changed ALT base
        motifs = engine.MotifSet(ctx, mats, cutoffs)
        ref_set = alt_set = None
        try:
            ref_set = dg.seqs.extract(cidx, cs, ce)
            t = ctx.timings()
            extract_ms = t["h2d"] + t["encode"]
            if variants.indels:
                ins_code = alt_code[np.repeat(first, a) + within]
                alt_set = dg.seqs.extract_splice(cidx, cs, ce, core_start, r, sub_off, ins_code)
            else:
                sub_pos = np.repeat(core_start, r) + within
                alt_set = dg.seqs.extract_subst(cidx, cs, ce, sub_off, sub_pos, alt_code)
            t = ctx.timings()
            extract_ms += t["h2d"] + t["encode"]
            if variants.indels:
                rows = engine.scan_variants_ex(ctx, motifs, ref_set, alt_set, core_start, r, a, st)
            else:
                rows = engine.scan_variants(ctx, motifs, ref_set, alt_set, core_start, r, st)
            t = ctx.timings()
        finally:
            for s in (ref_set, alt_set, motifs):
                if s is not None:
                    s.close()
    finally:
        if owned:
            dg.close()
    timings = {"extract": extract_ms, **{k: t[k] for k in ("prefilter", "exact", "order", "rows", "row_sort", "d2h")}}
    start = rows["start"].astype(np.int64) + cs[rows["allele"]]
    context_bp = int((ce - cs).sum())
    alt_bp = context_bp + int((a - r).sum())
    return VariantSites(n, n_motifs, rows["allele"], rows["motif"], start, rows["strand"], rows["ref_score"],
                        rows["alt_score"], rows["effect"] & 3, timings=timings, context_bp=context_bp,
                        motif_bp=(context_bp + alt_bp) * n_motifs, seconds=time.perf_counter() - t0,
                        paired=(rows["effect"] & 4) == 0)
