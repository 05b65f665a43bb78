"""Variant-effect scans: which motif sites do SNVs, MNVs and (opt-in) indels create or destroy (`motifscan variant`).

    variants = read_vcf("calls.vcf.gz", genome)          # alleles + skip counts; indels=True scans indels too
    sites = scan_variants(genome, pwms, cutoffs, variants)
    io.write_variant_tables(out_dir, pwms, variants, sites)

    variants = read_vcf("phased.vcf.gz", genome, indels=True, samples="all")
    sites = scan_haplotypes(genome, pwms, cutoffs, haplotype_clusters(variants, lmax))

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

Haplotypes (read_vcf(samples=...), haplotype_clusters, scan_haplotypes; `motifscan variant --haplotypes`): the phased
genotypes are read, and the alleles one haplotype carries within a motif width of each other form a cluster that is
scanned with all its changes applied, so alleles in cis that change a window together are scored together.  Identical
clusters are scanned once for all their carriers (DESIGN.md §5.5 has the rules).

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
CALL_SKIP_REASONS = ("missing", "unphased", "allele_skipped")
EFFECTS = {1: "loss", 2: "gain", 3: "both"}
STRAND = {"+": 1, "-": 2, "both": 3, 1: 1, 2: 2, 3: 3}

_CODE = np.full(256, 4, dtype=np.uint8)     # A/C/G/T in any case -> 0..3, every other byte -> 4 (cscore.c:91-110)
for _k, _b in enumerate(b"ACGT"):
    _CODE[_b] = _CODE[_b | 0x20] = _k


class Variants:
    """Alleles of a VCF, in input order.  Per allele: `chrom` (index into `chroms`), `pos` (0-based p = POS - 1),
    `ref`, `alt` and `id` as written in the file, and `record` (0-based index of its VCF record among the data lines).
    `skipped`: alleles left out, by reason; `n_records`: data lines read; `indels`: read with indels=True (the
    alleles may change the length, and scan_variants cuts every alt context with a splice).

    Genotypes (read_vcf(samples=...)): `samples` names the samples read; one call per (sample, haplotype) that carries
    a scanned allele: `call_allele` (index into the alleles), `call_sample` (index into `samples`) and `call_hap`
    (0 or 1).  `call_skipped`: calls left out, by reason (CALL_SKIP_REASONS)."""

    def __init__(self, chroms, chrom, pos, ref, alt, ids, record, skipped, n_records, indels=False, samples=(),
                 call_allele=(), call_sample=(), call_hap=(), call_skipped=None):
        self.indels = bool(indels)
        self.chroms = list(chroms)
        self.chrom = np.asarray(chrom, dtype=np.int32)
        self.pos = np.asarray(pos, dtype=np.int64)
        self.ref, self.alt, self.id = list(ref), list(alt), list(ids)
        self.record = np.asarray(record, dtype=np.int64)
        self.skipped = dict(skipped)
        self.n_records = int(n_records)
        self.samples = list(samples)
        self.call_allele = np.asarray(call_allele, dtype=np.int64)
        self.call_sample = np.asarray(call_sample, dtype=np.int32)
        self.call_hap = np.asarray(call_hap, dtype=np.int8)
        self.call_skipped = dict(call_skipped or dict.fromkeys(CALL_SKIP_REASONS, 0))

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


def read_vcf(path, genome, indels=False, samples=None):
    """The alleles of a VCF (see the module docstring for which are scanned) against `genome` (anything with
    `chroms` / `chrom_sizes`; REF is checked against its packed planes when it has them -- `PackedGenome`,
    `DeviceGenome` -- else against its fetched bases).  Lines starting with `#` are skipped; FILTER and INFO are
    ignored.  A data line with fewer than 5 tab-separated fields, or a POS that is not an integer, raises ValueError
    naming its line number.  `indels`: also scan alleles whose ALT length differs from REF's (else they count as
    `unsupported`).

    `samples`: None ignores the sample columns; "all" reads the genotypes of every sample named on the #CHROM line, a
    list those of the named ones (a name not in the header, or a VCF without sample columns, is a ValueError).  GT is
    parsed in Python, line by line (see _read_gt for the rules)."""
    chroms = list(genome.chroms)
    index = {c: i for i, c in enumerate(chroms)}
    sizes = [int(genome.chrom_sizes[c]) for c in chroms]
    skipped = dict.fromkeys(SKIP_REASONS, 0)
    chrom, pos, ref, alt, ids, record = [], [], [], [], [], []
    n_records = 0
    acgt = set("ACGTacgt")
    names, cols = [], None                   # the samples read and their columns (None: genotypes not read)
    calls = ([], [], [])                     # provisional allele (index into `chrom` ..., -1: not scanned), sample, hap
    call_skipped = dict.fromkeys(CALL_SKIP_REASONS, 0)
    with _open_text(path) as fh:
        for lineno, line in enumerate(fh, 1):
            if line.startswith("#"):
                if samples is not None and line.startswith("#CHROM"):
                    header = line.rstrip("\r\n").split("\t")[9:]
                    names = header if samples == "all" else list(dict.fromkeys(samples))
                    missing = [x for x in names if x not in header]
                    if missing:
                        raise ValueError(f"{path}: sample(s) not in the #CHROM line: {', '.join(missing)}")
                    cols = [9 + header.index(x) for x in names]
                continue
            line = line.rstrip("\r\n")
            if not line:
                continue
            f = line.split("\t", 5) if cols is None else line.split("\t")
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
            alt_index = []
            for a in f[4].split(","):
                if ci is None:
                    skipped["unknown_chrom"] += 1
                elif p < 0 or p + len(r) > sizes[ci]:
                    skipped["out_of_range"] += 1
                elif not a or not r or (len(a) != len(r) and not indels) or not acgt.issuperset(a):
                    skipped["unsupported"] += 1
                else:
                    alt_index.append(len(chrom))
                    chrom.append(ci)
                    pos.append(p)
                    ref.append(r)
                    alt.append(a)
                    ids.append(f[2])
                    record.append(rec)
                    continue
                alt_index.append(-1)
            if cols is not None:
                _read_gt(f, cols, alt_index, calls, call_skipped, f"{path}: line {lineno}")
    if samples is not None and not names:
        raise ValueError(f"{path}: no sample columns on the #CHROM line: no genotypes to read")
    chrom = np.array(chrom, dtype=np.int32)
    pos = np.array(pos, dtype=np.int64)
    ok = _ref_matches(genome, chrom, pos, ref)
    skipped["ref_mismatch"] = int((~ok).sum())
    keep = np.flatnonzero(ok)
    pick = keep.tolist()
    new_index = np.full(len(chrom) + 1, -1, dtype=np.int64)            # provisional -> final allele index; -1 stays
    new_index[keep] = np.arange(len(keep))
    call_allele = new_index[np.array(calls[0], dtype=np.int64)]
    scanned = call_allele >= 0
    call_skipped["allele_skipped"] += int((~scanned).sum())
    return Variants(chroms, chrom[keep], pos[keep], [ref[i] for i in pick], [alt[i] for i in pick],
                    [ids[i] for i in pick], np.array(record, dtype=np.int64)[keep] if record else np.zeros(0, np.int64),
                    skipped, n_records, indels=indels, samples=names, call_allele=call_allele[scanned],
                    call_sample=np.array(calls[1], dtype=np.int32)[scanned],
                    call_hap=np.array(calls[2], dtype=np.int8)[scanned], call_skipped=call_skipped)


def _read_gt(f, cols, alt_index, calls, skipped, where):
    """The genotype calls of one record (fields `f`) for the sample columns `cols`, appended to `calls` as
    (provisional allele index, sample, haplotype); `alt_index[k - 1]` is ALT k's provisional index (-1: not scanned).

    GT must be the first FORMAT key (VCF 4.x); when it is not, each sample's call counts once as `missing`.  `a|b`
    is phased: haplotype 0 carries ALT a and haplotype 1 ALT b.  An unphased `a/a` is unambiguous and both haplotypes
    carry it; each non-reference allele of an unphased heterozygous call counts as `unphased`.  A haploid `a` gives
    haplotype 0.  Each `.` allele counts as `missing`, each call to an ALT that is not scanned as `allele_skipped`;
    reference alleles (0) are not calls.  Ploidy above 2, or an allele index that is not an integer or above the
    record's ALT count, raises ValueError.  Phase sets (PS) are ignored: a `|` call is trusted."""
    has_gt = len(f) > 8 and f[8].split(":", 1)[0] == "GT"
    n_alts = len(alt_index)
    for si, col in enumerate(cols):
        if not has_gt or col >= len(f):
            skipped["missing"] += 1
            continue
        gt = f[col].split(":", 1)[0]
        if gt in ("0|0", "0/0", "0"):
            continue
        phased = "/" not in gt
        parts = gt.split("|") if phased else gt.split("/")
        if len(parts) > 2:
            raise ValueError(f"{where}: sample column {col + 1}: GT {gt!r} has ploidy {len(parts)}; at most 2 is read")
        idx = []
        for x in parts:
            if x == ".":
                idx.append(None)
                continue
            try:
                k = int(x)
            except ValueError:
                raise ValueError(f"{where}: sample column {col + 1}: GT allele {x!r} is not an integer") from None
            if k < 0 or k > n_alts:
                raise ValueError(f"{where}: sample column {col + 1}: GT allele {k} but the record has {n_alts} ALT")
            idx.append(k)
        if not phased and idx[0] != idx[1]:
            for k in idx:
                if k is None:
                    skipped["missing"] += 1
                elif k:
                    skipped["unphased"] += 1
            continue
        for h, k in enumerate(idx):
            if k is None:
                skipped["missing"] += 1
            elif k:
                calls[0].append(alt_index[k - 1])
                calls[1].append(si)
                calls[2].append(h)


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


def _changes(variants):
    """Per allele (p, r, first, a): r reference bases at p replaced by the a ALT bytes from `first` on of the
    concatenated ALTs -- _trim's change in indel mode, the untrimmed allele otherwise."""
    if variants.indels:
        return _trim(variants)
    r = np.fromiter((len(x) for x in variants.ref), dtype=np.int64, count=len(variants))
    return variants.pos, r, np.cumsum(r) - r, r


class Haplotypes:
    """The distinct allele clusters that the phased haplotypes of `variants` carry (haplotype_clusters).  Cluster c
    lies on chromosome `chrom[c]` (index into variants.chroms) and holds the alleles `allele[allele_off[c] ..
    allele_off[c + 1])` (indices into `variants`) in change order; its carriers are (`carrier_sample`, `carrier_hap`)
    [carrier_off[c] .. carrier_off[c + 1]) in (sample, haplotype) order.  `overlap`: calls dropped because their
    change conflicts with an earlier one on the same haplotype; `lmax`: the longest motif the clusters are exact for.
    `p`, `r`, `a`, `first`: every allele's change (_changes)."""

    def __init__(self, variants, lmax, chrom, allele_off, allele, carrier_off, carrier_sample, carrier_hap, overlap):
        self.variants, self.lmax = variants, int(lmax)
        self.chrom = np.asarray(chrom, dtype=np.int32)
        self.allele_off, self.allele = np.asarray(allele_off, dtype=np.int64), np.asarray(allele, dtype=np.int64)
        self.carrier_off = np.asarray(carrier_off, dtype=np.int64)
        self.carrier_sample = np.asarray(carrier_sample, dtype=np.int32)
        self.carrier_hap = np.asarray(carrier_hap, dtype=np.int8)
        self.overlap = int(overlap)
        self.p, self.r, self.first, self.a = _changes(variants)

    def __len__(self):
        return len(self.chrom)

    def sizes(self):
        """Alleles per cluster."""
        return np.diff(self.allele_off)


def haplotype_clusters(variants, lmax):
    """Cluster the alleles each phased haplotype of `variants` (read_vcf(samples=...)) carries, for motifs of at most
    `lmax` bases.  Per (sample, haplotype, chromosome) the alleles are sorted by their change (p, r) (_changes: trimmed
    in indel mode) and the allele index.  A change that starts before the last kept one ends, p2 < p1 + max(r1, 1)
    (an insertion occupies its junction), conflicts: it is dropped from that haplotype and counted as `overlap`.
    Consecutive kept changes join one cluster when p2 - (p1 + r1) <= lmax - 2; with a larger gap no window of any
    motif touches both, so scanning them apart is exact.  Clusters are identified by their tuple of alleles,
    de-duplicated across samples and haplotypes (a single allele is a cluster too) and numbered by chromosome (genome
    order), first change, then allele tuple."""
    p, r, _, _ = _changes(variants)
    al = variants.call_allele
    hap = variants.call_sample.astype(np.int64) * 2 + variants.call_hap
    ch = variants.chrom[al].astype(np.int64)
    cp, cr = p[al], r[al]
    order = np.lexsort((al, cr, cp, ch, hap))
    al, hap, ch, cp, cr = al[order], hap[order], ch[order], cp[order], cr[order]
    end = cp + np.maximum(cr, 1)
    keep = np.ones(len(al), dtype=bool)
    while True:                                       # conflicts with the previous kept change, first of each run
        k = np.flatnonzero(keep)
        same = (hap[k][1:] == hap[k][:-1]) & (ch[k][1:] == ch[k][:-1])
        conflict = np.zeros(len(k), dtype=bool)
        conflict[1:] = same & (cp[k][1:] < end[k][:-1])
        first = conflict & ~np.r_[False, conflict[:-1]]
        if not first.any():
            break
        keep[k[first]] = False
    overlap = int((~keep).sum())
    al, hap, ch, cp, cr = al[keep], hap[keep], ch[keep], cp[keep], cr[keep]
    new = np.ones(len(al), dtype=bool)
    new[1:] = (hap[1:] != hap[:-1]) | (ch[1:] != ch[:-1]) | (cp[1:] - (cp[:-1] + cr[:-1]) > lmax - 2)
    hc_first = np.flatnonzero(new)                    # haplotype clusters: [hc_first[i], hc_first[i + 1])
    hc_size = np.diff(np.r_[hc_first, len(al)])
    # de-duplicate by allele tuple, one size at a time
    tuples, hc_distinct = [], np.zeros(len(hc_first), dtype=np.int64)
    for k in np.unique(hc_size).tolist():
        sel = np.flatnonzero(hc_size == k)
        rows = al[hc_first[sel][:, None] + np.arange(k)]
        uniq, inv = np.unique(rows, axis=0, return_inverse=True)
        hc_distinct[sel] = len(tuples) + inv.reshape(-1)
        tuples.extend(tuple(t) for t in uniq.tolist())
    rank = sorted(range(len(tuples)), key=lambda d: (int(variants.chrom[tuples[d][0]]), int(p[tuples[d][0]]),
                                                     int(r[tuples[d][0]]), tuples[d]))
    number = np.empty(len(tuples), dtype=np.int64)
    number[rank] = np.arange(len(tuples))
    tuples = [tuples[d] for d in rank]
    sizes = np.array([len(t) for t in tuples], dtype=np.int64)
    allele_off = np.zeros(len(tuples) + 1, dtype=np.int64)
    np.cumsum(sizes, out=allele_off[1:])
    allele = np.array([a for t in tuples for a in t], dtype=np.int64)
    chrom = variants.chrom[allele[allele_off[:-1]]] if len(tuples) else np.zeros(0, np.int32)
    cl = number[hc_distinct]
    hc_hap = hap[hc_first]
    o = np.lexsort((hc_hap, cl))
    carrier_off = np.zeros(len(tuples) + 1, dtype=np.int64)
    np.cumsum(np.bincount(cl, minlength=len(tuples)), out=carrier_off[1:])
    return Haplotypes(variants, lmax, chrom, allele_off, allele, carrier_off, hc_hap[o] // 2, hc_hap[o] % 2, overlap)


class HaplotypeSites:
    """Rows of a haplotype scan in (cluster, motif, own-side start, strand, ref before alt) order -- the own side is
    the alt haplotype for a gain and the reference otherwise: `cluster`, `motif`, `strand` (1 / 2), `ref_start` (the
    window's start on the chromosome, -1 when it has none there), `alt_start` (its start on the haplotype, numbered
    like the chromosome left of the cluster's first change; -1 when it has none there), `ref_score` / `alt_score`,
    `effect` (1 loss, 2 gain, 3 both) and `paired` (false when the window exists on one side only: the other score is
    NaN).  `timings`, `context_bp`, `motif_bp` and `seconds` as in VariantSites.  `carrier_off` / `carrier_id`: the
    haplotypes (sample * 2 + haplotype) carrying each cluster, for summary()."""

    def __init__(self, n_clusters, n_motifs, cluster, motif, strand, ref_start, alt_start, ref_score, alt_score, effect,
                 paired, carrier_off=None, carrier_id=None, timings=None, context_bp=0, motif_bp=0, seconds=0.0):
        self.n_clusters, self.n_motifs = int(n_clusters), int(n_motifs)
        self.cluster, self.motif = np.asarray(cluster, dtype=np.int32), np.asarray(motif, dtype=np.int32)
        self.strand = np.asarray(strand, dtype=np.int8)
        self.ref_start, self.alt_start = np.asarray(ref_start, dtype=np.int64), np.asarray(alt_start, dtype=np.int64)
        self.ref_score, self.alt_score = np.asarray(ref_score, dtype=np.float64), np.asarray(alt_score, dtype=np.float64)
        self.effect = np.asarray(effect, dtype=np.int8)
        self.paired = np.asarray(paired, dtype=bool)
        self.carrier_off = np.zeros(self.n_clusters + 1, np.int64) if carrier_off is None else np.asarray(carrier_off)
        self.carrier_id = np.zeros(0, np.int64) if carrier_id is None else np.asarray(carrier_id, dtype=np.int64)
        self.timings = dict(timings or {})
        self.context_bp, self.motif_bp, self.seconds = int(context_bp), int(motif_bp), float(seconds)

    def __len__(self):
        return len(self.cluster)

    def rows_by_effect(self):
        return {name: int((self.effect == code).sum()) for code, name in EFFECTS.items()}

    def summary(self):
        """Per motif (set order), the clusters with at least one row of each effect (n_gain, n_loss, n_both) and the
        distinct haplotypes that carry such a cluster (hap_gain, hap_loss, hap_both): dict of int64 arrays."""
        out = {}
        n_c = max(self.n_clusters, 1)
        for code, name in ((2, "gain"), (1, "loss"), (3, "both")):
            sel = self.effect == code
            pairs = np.unique(self.motif[sel].astype(np.int64) * n_c + self.cluster[sel])
            m, c = pairs // n_c, pairs % n_c
            out["n_" + name] = np.bincount(m, minlength=self.n_motifs).astype(np.int64)
            cnt = self.carrier_off[c + 1] - self.carrier_off[c]
            at = np.repeat(self.carrier_off[c] - np.cumsum(cnt) + cnt, cnt) + np.arange(int(cnt.sum()))
            mh = np.unique(np.repeat(m, cnt) * (int(self.carrier_id.max(initial=0)) + 1) + self.carrier_id[at])
            out["hap_" + name] = np.bincount(mh // (int(self.carrier_id.max(initial=0)) + 1),
                                             minlength=self.n_motifs).astype(np.int64)
        return out


def scan_haplotypes(genome, pwms, cutoffs, haplotypes, strand="both", device=0):
    """Rows of every cluster of `haplotypes` (haplotype_clusters) for the motif set `pwms` at `cutoffs`, on one GPU
    (`genome` as in scan_variants).  Cluster c's ref context is [max(p_first - Lmax + 1, 0), min(p_last + r_last +
    Lmax - 1, size)) of its chromosome; its alt context is the same interval with every allele's change applied
    (msb_seqs_extract_edits); msb_scan_haplotypes keeps the windows that touch a change on their own side and pairs
    them across the edits.  The clusters go to the device in batches whose row keys fit 64 bits."""
    mats = [np.asarray(getattr(p, "matrix", p), dtype=np.float64) for p in pwms]
    n, n_motifs = len(haplotypes), len(mats)
    st = STRAND[strand]
    h = haplotypes
    carrier_id = h.carrier_sample.astype(np.int64) * 2 + h.carrier_hap
    if n == 0 or n_motifs == 0:
        e = np.zeros(0)
        return HaplotypeSites(n, n_motifs, e, e, e, e, e, e, e, e, e, h.carrier_off, carrier_id)
    lmax = max(m.shape[1] for m in mats)
    if lmax > h.lmax:
        raise ValueError(f"the clusters were built for motifs of at most {h.lmax} bases, the longest has {lmax}")
    t0 = time.perf_counter()
    v = h.variants
    dg, owned = _device_genome(genome, device)
    timings = dict.fromkeys(("extract", "prefilter", "exact", "order", "rows", "row_sort", "d2h"), 0.0)
    parts = []
    try:
        ctx = dg.ctx
        cidx = np.array([dg.chrom_index[c] for c in v.chroms], dtype=np.int32)[h.chrom]
        size = np.array([dg.chrom_sizes[c] for c in dg.chroms], dtype=np.int64)[cidx]
        al = h.allele
        first, last = al[h.allele_off[:-1]], al[h.allele_off[1:] - 1]
        cs = np.maximum(h.p[first] - (lmax - 1), 0)
        ce = np.minimum(h.p[last] + h.r[last] + lmax - 1, size)
        counts = np.diff(h.allele_off)
        edit_at = h.p[al] - np.repeat(cs, counts)
        edit_r, edit_a = h.r[al], h.a[al]
        alt_code = _CODE[np.frombuffer("".join(v.alt).encode("ascii"), dtype=np.uint8)]
        ins_off = np.zeros(len(al) + 1, dtype=np.int64)
        np.cumsum(edit_a, out=ins_off[1:])
        within = np.arange(int(ins_off[-1]), dtype=np.int64) - np.repeat(ins_off[:-1], edit_a)
        ins_code = alt_code[np.repeat(h.first[al], edit_a) + within]
        net = np.add.reduceat(edit_a - edit_r, h.allele_off[:-1])
        bits = lambda x: int(x - 1).bit_length() if x > 1 else 0            # noqa: E731
        per = 1 << max(62 - bits(n_motifs) - bits(int(max((ce - cs).max(), (ce - cs + net).max()))), 0)
        motifs = engine.MotifSet(ctx, mats, cutoffs)
        try:
            for b0 in range(0, n, per):
                b1 = min(n, b0 + per)
                e0, e1 = int(h.allele_off[b0]), int(h.allele_off[b1])
                ref_set = alt_set = None
                try:
                    ref_set = dg.seqs.extract(cidx[b0:b1], cs[b0:b1], ce[b0:b1])
                    t = ctx.timings()
                    timings["extract"] += t["h2d"] + t["encode"]
                    alt_set = dg.seqs.extract_edits(cidx[b0:b1], cs[b0:b1], ce[b0:b1], h.allele_off[b0:b1 + 1] - e0,
                                                    edit_at[e0:e1], edit_r[e0:e1], ins_off[e0:e1 + 1] - ins_off[e0],
                                                    ins_code[ins_off[e0]:ins_off[e1]])
                    t = ctx.timings()
                    timings["extract"] += t["h2d"] + t["encode"]
                    rows = engine.scan_haplotypes(ctx, motifs, ref_set, alt_set, h.allele_off[b0:b1 + 1] - e0,
                                                  edit_at[e0:e1], edit_r[e0:e1], edit_a[e0:e1], st)
                    t = ctx.timings()
                    for k in ("prefilter", "exact", "order", "rows", "row_sort", "d2h"):
                        timings[k] += t[k]
                    rows["context"] = rows["context"].astype(np.int64) + b0
                    parts.append(rows)
                finally:
                    for s in (ref_set, alt_set):
                        if s is not None:
                            s.close()
        finally:
            motifs.close()
    finally:
        if owned:
            dg.close()
    rows = {k: np.concatenate([r[k] for r in parts]) for k in parts[0]}
    c = rows["context"]
    eff = rows["effect"]
    from_alt = (eff & 3) == 2
    own, other = rows["start"].astype(np.int64), rows["other_start"].astype(np.int64)
    ref_rel, alt_rel = np.where(from_alt, other, own), np.where(from_alt, own, other)
    context_bp = int((ce - cs).sum())
    alt_bp = context_bp + int(net.sum())
    return HaplotypeSites(n, n_motifs, c, rows["motif"], rows["strand"], np.where(ref_rel >= 0, ref_rel + cs[c], -1),
                          np.where(alt_rel >= 0, alt_rel + cs[c], -1), rows["ref_score"], rows["alt_score"], eff & 3,
                          (eff & 4) == 0, h.carrier_off, carrier_id, timings=timings, context_bp=context_bp,
                          motif_bp=(context_bp + alt_bp) * n_motifs, seconds=time.perf_counter() - t0)
