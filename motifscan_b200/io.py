"""Result writers of `motifscan scan` (reference motifscan/io/__init__.py:12-71): same file names,
columns and number formatting (`str()` of ints and Python floats), fed from the scan's arrays.

    motif_sites_number.xls   chr, 1-based start, end, then the site count per motif
    motif_sites_score.xls    same header, the best score per motif or `NA`
    motif_sites/<id>_<name>_sites.bed   chrom, site start, start + L, '.', score, strand
    motif_enrichment.xls     sorted by (enriched p-value, -fold change)
    motif_variant_sites.xls / motif_variant_summary.xls   `motifscan variant` (write_variant_tables)
    motif_centrality.xls / motif_site_distribution.xls   `scan --centrality` (write_centrality_tables)
"""
import os
import re

import numpy as np


def replace_special_char(name):
    """Motif name as a file name (reference io/utils.py:15-16): `-`, `:`, `.`, `/`, `*` -> `_`."""
    return re.sub(r"[-:./*]", "_", name)


def _motif_names(pwms, sep=","):
    return [f"{pwm.matrix_id}{sep}{pwm.name}" for pwm in pwms]


def _cell_tables(motif_sites, n_pwms, n_regions):
    """(counts int64[n_regions, n_pwms], best float64[n_regions, n_pwms] with NaN where empty)."""
    counts = np.zeros((n_regions, n_pwms), dtype=np.int64)
    best = np.full((n_regions, n_pwms), np.nan)
    if hasattr(motif_sites, "_off"):     # MotifSites: sites sorted by (motif, region)
        for m in range(n_pwms):
            a, b = int(motif_sites._off[m]), int(motif_sites._off[m + 1])
            if b > a:
                seq = motif_sites._seq_idx[a:b]
                np.add.at(counts[:, m], seq, 1)
                col = np.full(n_regions, -np.inf)
                np.maximum.at(col, seq, motif_sites._score[a:b])
                hit = counts[:, m] > 0
                best[hit, m] = col[hit]
    else:
        for m, per_motif in enumerate(motif_sites):
            for r, cell in enumerate(per_motif):
                counts[r, m] = len(cell)
                if cell:
                    best[r, m] = max(site.score for site in cell)
    return counts, best


def _write_sites_table_blocks(f_num, f_score, regions, motif_sites, n_pwms, block_rows=8192):
    """The two tables block by block from the scan's arrays: the cells of a block of rows are filled and
    formatted by the library on host threads (msb_format_site_tables; numbers look like Python's str()), so
    200,000 regions x 1,900 motifs never exist as a dense table, let alone as Python objects."""
    import ctypes
    from . import _lib
    lib = _lib.load()
    off = np.ascontiguousarray(motif_sites._off, dtype=np.int64)
    seq = np.ascontiguousarray(motif_sites._seq_idx, dtype=np.int32)
    score = np.ascontiguousarray(motif_sites._score, dtype=np.float64)
    if seq.size == 0:
        seq, score = np.zeros(1, np.int32), np.zeros(1, np.float64)
    n_threads = min(os.cpu_count() or 1, 32)
    for r0 in range(0, len(regions), block_rows):
        r1 = min(r0 + block_rows, len(regions))
        leads = [f"{g.chrom}\t{g.start + 1}\t{g.end}\t".encode() for g in regions[r0:r1]]
        lead_off = np.zeros(len(leads) + 1, dtype=np.int64)
        np.cumsum([len(x) for x in leads], out=lead_off[1:])
        p_num, p_score = ctypes.c_void_p(), ctypes.c_void_p()
        n_num, n_score = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(lib.msb_format_site_tables(n_pwms, _lib.ptr(off, ctypes.c_int64), _lib.ptr(seq, ctypes.c_int32),
                                              _lib.ptr(score, ctypes.c_double), r0, r1, b"".join(leads),
                                              _lib.ptr(lead_off, ctypes.c_int64), ctypes.byref(p_num), ctypes.byref(n_num),
                                              ctypes.byref(p_score), ctypes.byref(n_score), n_threads))
        try:
            # straight from the library's buffers to the files, no copy into a bytes object
            f_num.write((ctypes.c_char * n_num.value).from_address(p_num.value))
            f_score.write((ctypes.c_char * n_score.value).from_address(p_score.value))
        finally:
            lib.msb_text_free(p_num)
            lib.msb_text_free(p_score)


def write_sites_table(output_dir, pwms, regions, motif_sites):
    os.makedirs(output_dir, exist_ok=True)
    header = "chr\tstart\tend\t" + "\t".join(_motif_names(pwms)) + "\n"
    if hasattr(motif_sites, "_off"):     # a scan's arrays: streamed through the native formatter
        with open(os.path.join(output_dir, "motif_sites_number.xls"), "wb") as f_num, \
                open(os.path.join(output_dir, "motif_sites_score.xls"), "wb") as f_score:
            f_num.write(header.encode())
            f_score.write(header.encode())
            _write_sites_table_blocks(f_num, f_score, list(regions), motif_sites, len(pwms))
        return
    counts, best = _cell_tables(motif_sites, len(pwms), len(regions))
    with open(os.path.join(output_dir, "motif_sites_number.xls"), "w") as f_num, \
            open(os.path.join(output_dir, "motif_sites_score.xls"), "w") as f_score:
        f_num.write(header)
        f_score.write(header)
        for r, region in enumerate(regions):
            lead = f"{region.chrom}\t{region.start + 1}\t{region.end}\t"
            f_num.write(lead + "\t".join(map(str, counts[r].tolist())) + "\n")
            row = best[r].tolist()
            f_score.write(lead + "\t".join("NA" if c == 0 else str(v) for c, v in zip(counts[r].tolist(), row)) + "\n")


def write_cell_tables(output_dir, pwms, regions, counts, best):
    """The two tables from per-cell statistics: `counts` / `best` [n_regions, n_motifs] (a whole-genome scan's
    per-(chromosome, motif) counts and best scores), formatted by the library (msb_format_cell_tables)."""
    import ctypes
    from . import _lib
    lib = _lib.load()
    os.makedirs(output_dir, exist_ok=True)
    header = ("chr\tstart\tend\t" + "\t".join(_motif_names(pwms)) + "\n").encode()
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    best = np.ascontiguousarray(best, dtype=np.float64)
    leads = [f"{g.chrom}\t{g.start + 1}\t{g.end}\t".encode() for g in regions]
    lead_off = np.zeros(len(leads) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in leads], out=lead_off[1:])
    p_num, p_score = ctypes.c_void_p(), ctypes.c_void_p()
    n_num, n_score = ctypes.c_int64(0), ctypes.c_int64(0)
    _lib.check(lib.msb_format_cell_tables(len(leads), len(pwms), _lib.ptr(counts, ctypes.c_int64), _lib.ptr(best, ctypes.c_double),
                                          b"".join(leads), _lib.ptr(lead_off, ctypes.c_int64), ctypes.byref(p_num),
                                          ctypes.byref(n_num), ctypes.byref(p_score), ctypes.byref(n_score),
                                          min(os.cpu_count() or 1, 32)))
    try:
        with open(os.path.join(output_dir, "motif_sites_number.xls"), "wb") as f_num, \
                open(os.path.join(output_dir, "motif_sites_score.xls"), "wb") as f_score:
            f_num.write(header)
            f_score.write(header)
            if n_num.value:
                f_num.write((ctypes.c_char * n_num.value).from_address(p_num.value))
                f_score.write((ctypes.c_char * n_score.value).from_address(p_score.value))
    finally:
        lib.msb_text_free(p_num)
        lib.msb_text_free(p_score)


def _site_arrays(motif_sites, regions):
    """(offsets, group, start, group_base or None, score, strand, group names) of an array-backed result: the
    `MotifSites` of a region scan (groups = regions, starts relative to the region's scan window) or the
    `GenomeSites` of a whole-genome scan (groups = chromosomes, starts on the chromosome); None otherwise."""
    if hasattr(motif_sites, "_off"):
        base = np.asarray(motif_sites.seq_starts, dtype=np.int64)
        return (motif_sites._off, motif_sites._seq_idx, motif_sites._start, base, motif_sites._score, motif_sites._strand,
                [g.chrom for g in regions])
    if hasattr(motif_sites, "chrom_idx"):
        return (motif_sites.offsets, motif_sites.chrom_idx, motif_sites.start, None, motif_sites.score, motif_sites.strand,
                list(motif_sites.chroms))
    return None


def write_sites_bed(output_dir, pwms, regions, motif_sites):
    """One BED file per motif.  Array-backed results are formatted by the library on host threads and written in
    blocks (msb_write_sites_bed, numbers like Python's str()); nested lists are written line by line."""
    out_dir = os.path.join(output_dir, "motif_sites")
    os.makedirs(out_dir, exist_ok=True)
    arrays = _site_arrays(motif_sites, regions)
    if arrays is not None:
        import ctypes
        from . import _lib
        lib = _lib.load()
        off, group, start, base, score, strand, names = arrays
        group = np.ascontiguousarray(group, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        score = np.ascontiguousarray(score, dtype=np.float64)
        strand = np.ascontiguousarray(strand, dtype=np.int8)
        enc = [x.encode() for x in names]
        name_off = np.zeros(len(enc) + 1, dtype=np.int64)
        np.cumsum([len(x) for x in enc], out=name_off[1:])
        n_threads = min(os.cpu_count() or 1, 32)
        for m, pwm in enumerate(pwms):
            path = os.path.join(out_dir, replace_special_char(f"{pwm.matrix_id}_{pwm.name}") + "_sites.bed")
            a, b = int(off[m]), int(off[m + 1])
            _lib.check(lib.msb_write_sites_bed(
                path.encode(), b - a, _lib.ptr(group[a:], ctypes.c_int32) if b > a else None,
                _lib.ptr(start[a:], ctypes.c_int32) if b > a else None, _lib.ptr(base, ctypes.c_int64) if base is not None else None,
                _lib.ptr(score[a:], ctypes.c_double) if b > a else None, _lib.ptr(strand[a:], ctypes.c_int8) if b > a else None,
                int(pwm.length), len(enc), b"".join(enc), _lib.ptr(name_off, ctypes.c_int64), n_threads))
        return
    for pwm, per_motif in zip(pwms, motif_sites):
        path = os.path.join(out_dir, replace_special_char(f"{pwm.matrix_id}_{pwm.name}") + "_sites.bed")
        with open(path, "w") as out:
            for region, cell in zip(regions, per_motif):
                for site in cell:
                    out.write(f"{region.chrom}\t{site.start}\t{site.start + pwm.length}\t.\t{site.score}\t{site.strand}\n")


VARIANT_SITES_HEADER = ("chrom\tpos\tid\tref\talt\tmotif_id\tmotif_name\tstart\tend\tstrand\tref_score\talt_score\t"
                        "effect\n")
VARIANT_SUMMARY_HEADER = "motif_id\tmotif_name\tn_gain\tn_loss\tn_both\n"


def write_variant_tables(output_dir, pwms, variants, sites):
    """The two tables of `motifscan variant` (variants.scan_variants):

        motif_variant_sites.xls    one row per (allele, motif, window, strand) that is a site on at least one allele:
                                   chrom, pos, id, ref and alt as in the VCF (alt = the allele), motif id and name,
                                   the window [start, end) 0-based half-open on the allele's haplotype, strand,
                                   both scores (NA where an indel leaves no window on that allele) and the effect
        motif_variant_summary.xls  per motif, the alleles with at least one gain / loss / both row

    The site rows are formatted by the library on host threads (msb_write_variant_table; scores like Python's
    str()), so tens of millions of rows never become Python objects."""
    import ctypes
    from . import _lib
    lib = _lib.load()
    os.makedirs(output_dir, exist_ok=True)
    allele = np.ascontiguousarray(sites.allele, dtype=np.int32)
    used, row_allele = np.unique(allele, return_inverse=True)          # leads only for alleles with a row
    row_allele = np.ascontiguousarray(row_allele, dtype=np.int32)
    leads = [f"{variants.chroms[variants.chrom[a]]}\t{int(variants.pos[a]) + 1}\t{variants.id[a]}\t{variants.ref[a]}\t"
             f"{variants.alt[a]}\t".encode() for a in used.tolist()]
    lead_off = np.zeros(len(leads) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in leads], out=lead_off[1:])
    mtext = [f"{pwm.matrix_id}\t{pwm.name}\t".encode() for pwm in pwms]
    motif_off = np.zeros(len(mtext) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in mtext], out=motif_off[1:])
    motif_len = np.array([int(pwm.length) for pwm in pwms] or [0], dtype=np.int32)
    n = len(allele)
    motif = np.ascontiguousarray(sites.motif, dtype=np.int32)
    start = np.ascontiguousarray(sites.start, dtype=np.int32)
    strand = np.ascontiguousarray(sites.strand, dtype=np.int8)
    ref_score = np.ascontiguousarray(sites.ref_score, dtype=np.float64)
    alt_score = np.ascontiguousarray(sites.alt_score, dtype=np.float64)
    effect = np.ascontiguousarray(np.where(sites.paired, sites.effect, sites.effect | 4), dtype=np.int8)
    arrays = [(row_allele, ctypes.c_int32), (motif, ctypes.c_int32), (start, ctypes.c_int32), (strand, ctypes.c_int8),
              (ref_score, ctypes.c_double), (alt_score, ctypes.c_double), (effect, ctypes.c_int8)]
    _lib.check(lib.msb_write_variant_table(
        os.path.join(output_dir, "motif_variant_sites.xls").encode(), VARIANT_SITES_HEADER.encode(), n,
        *[_lib.ptr(a, ct) if n else None for a, ct in arrays], len(leads), b"".join(leads),
        _lib.ptr(lead_off, ctypes.c_int64), len(pwms), b"".join(mtext), _lib.ptr(motif_off, ctypes.c_int64),
        _lib.ptr(motif_len, ctypes.c_int32), min(os.cpu_count() or 1, 32)))
    summary = sites.summary()
    with open(os.path.join(output_dir, "motif_variant_summary.xls"), "w") as out:
        out.write(VARIANT_SUMMARY_HEADER)
        for m, pwm in enumerate(pwms):
            out.write(f"{pwm.matrix_id}\t{pwm.name}\t{int(summary['n_gain'][m])}\t{int(summary['n_loss'][m])}\t"
                      f"{int(summary['n_both'][m])}\n")


HAPLOTYPE_SITES_HEADER = ("chrom\tcluster\tids\tmotif_id\tmotif_name\tref_start\tref_end\talt_start\talt_end\tstrand\t"
                          "ref_score\talt_score\teffect\n")
HAPLOTYPE_CLUSTERS_HEADER = "cluster\tchrom\talleles\tids\tcarriers\n"
HAPLOTYPE_SUMMARY_HEADER = "motif_id\tmotif_name\tn_gain\tn_loss\tn_both\thap_gain\thap_loss\thap_both\n"


def write_haplotype_tables(output_dir, pwms, haplotypes, sites):
    """The three tables of `motifscan variant --haplotypes` (variants.scan_haplotypes):

        motif_haplotype_sites.xls     one row per (cluster, motif, window pair, strand) that is a site on at least one
                                      side: chrom, cluster, the alleles' IDs (comma-separated), motif id and name, the
                                      window on the chromosome [ref_start, ref_end) and on the haplotype [alt_start,
                                      alt_end) (0-based half-open; NA NA where it has none), strand, both scores (NA
                                      where there is no window) and the effect
        motif_haplotype_clusters.xls  per cluster: chrom, its alleles as POS:REF>ALT and their IDs (comma-separated),
                                      and its carriers as sample:1 / sample:2 (first / second haplotype)
        motif_haplotype_summary.xls   per motif, the clusters with at least one gain / loss / both row and the
                                      haplotypes that carry such a cluster

    The site rows are formatted by the library on host threads (msb_write_haplotype_table, shared with
    msb_write_variant_table)."""
    import ctypes
    from . import _lib
    lib = _lib.load()
    os.makedirs(output_dir, exist_ok=True)
    v, h = haplotypes.variants, haplotypes
    ids = [",".join(v.id[a] for a in h.allele[h.allele_off[c]:h.allele_off[c + 1]].tolist()) for c in range(len(h))]
    cluster = np.ascontiguousarray(sites.cluster, dtype=np.int32)
    used, row_cluster = np.unique(cluster, return_inverse=True)        # leads only for clusters with a row
    row_cluster = np.ascontiguousarray(row_cluster.reshape(-1), dtype=np.int32)
    leads = [f"{v.chroms[h.chrom[c]]}\t{c}\t{ids[c]}\t".encode() for c in used.tolist()]
    lead_off = np.zeros(len(leads) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in leads], out=lead_off[1:])
    mtext = [f"{pwm.matrix_id}\t{pwm.name}\t".encode() for pwm in pwms]
    motif_off = np.zeros(len(mtext) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in mtext], out=motif_off[1:])
    motif_len = np.array([int(pwm.length) for pwm in pwms] or [0], dtype=np.int32)
    n = len(cluster)
    arrays = [(row_cluster, ctypes.c_int32), (np.ascontiguousarray(sites.motif, dtype=np.int32), ctypes.c_int32),
              (np.ascontiguousarray(sites.ref_start, dtype=np.int64), ctypes.c_int64),
              (np.ascontiguousarray(sites.alt_start, dtype=np.int64), ctypes.c_int64),
              (np.ascontiguousarray(sites.strand, dtype=np.int8), ctypes.c_int8),
              (np.ascontiguousarray(sites.ref_score, dtype=np.float64), ctypes.c_double),
              (np.ascontiguousarray(sites.alt_score, dtype=np.float64), ctypes.c_double),
              (np.ascontiguousarray(np.where(sites.paired, sites.effect, sites.effect | 4), dtype=np.int8), ctypes.c_int8)]
    _lib.check(lib.msb_write_haplotype_table(
        os.path.join(output_dir, "motif_haplotype_sites.xls").encode(), HAPLOTYPE_SITES_HEADER.encode(), n,
        *[_lib.ptr(a, ct) if n else None for a, ct in arrays], len(leads), b"".join(leads),
        _lib.ptr(lead_off, ctypes.c_int64), len(pwms), b"".join(mtext), _lib.ptr(motif_off, ctypes.c_int64),
        _lib.ptr(motif_len, ctypes.c_int32), min(os.cpu_count() or 1, 32)))
    with open(os.path.join(output_dir, "motif_haplotype_clusters.xls"), "w") as out:
        out.write(HAPLOTYPE_CLUSTERS_HEADER)
        for c in range(len(h)):
            alleles = ",".join(f"{int(v.pos[a]) + 1}:{v.ref[a]}>{v.alt[a]}"
                               for a in h.allele[h.allele_off[c]:h.allele_off[c + 1]].tolist())
            k0, k1 = int(h.carrier_off[c]), int(h.carrier_off[c + 1])
            carriers = ",".join(f"{v.samples[s]}:{x + 1}" for s, x in zip(h.carrier_sample[k0:k1].tolist(),
                                                                           h.carrier_hap[k0:k1].tolist()))
            out.write(f"{c}\t{v.chroms[h.chrom[c]]}\t{alleles}\t{ids[c]}\t{carriers}\n")
    summary = sites.summary()
    with open(os.path.join(output_dir, "motif_haplotype_summary.xls"), "w") as out:
        out.write(HAPLOTYPE_SUMMARY_HEADER)
        for m, pwm in enumerate(pwms):
            out.write(f"{pwm.matrix_id}\t{pwm.name}\t" + "\t".join(
                str(int(summary[k][m])) for k in ("n_gain", "n_loss", "n_both", "hap_gain", "hap_loss", "hap_both")) + "\n")


def write_enrich_table(output_dir, enrichment_results):
    os.makedirs(output_dir, exist_ok=True)
    enrichment_results.sort(key=lambda res: (res.p_enriched, -res.fold_change))   # io/__init__.py:63
    with open(os.path.join(output_dir, "motif_enrichment.xls"), "w") as out:
        out.write("Motif\tNum_input_regions\tNum_control_regions\tFold_change\tEnriched_P_value\t"
                  "Depleted_P_value\tCorrected_P_value\n")
        for res in enrichment_results:
            out.write(f"{res.name}\t{res.n_input}\t{res.n_control}\t{res.fold_change}\t{res.p_enriched}\t"
                      f"{res.p_depleted}\t{res.p_corrected}\n")


COOCCUR_HEADER = ("Motif_A\tMotif_B\tNum_A\tNum_B\tNum_both\tExpected\tRatio\tP_cooccur\tP_exclusive\tCorrected_P_value\t"
                  "Num_both_control\tFold_change\tEnriched_P_value\tDepleted_P_value\tCorrected_enriched_P_value\n")
SPACING_HEADER = "Anchor\tPartner\tOrientation\tPairs\tPeak_offset\tPeak_pairs\tExpected\tP_value\tCounts\n"


def write_cooccur_table(output_dir, pwms, table):
    """motif_cooccurrence.xls: one row per motif pair a < b (cooccur.cooccur_table), mutually exclusive pairs included,
    ordered by (P_cooccur, -Ratio, a, b); motifs as `matrix_id,name`, numbers like Python's str(), the control columns
    `NA` without controls.  Millions of rows are formatted by the library on host threads (msb_write_cooccur_table)."""
    import ctypes
    from . import _lib
    from .cooccur import cooccur_order
    lib = _lib.load()
    os.makedirs(output_dir, exist_ok=True)
    order = cooccur_order(table)
    mtext = [name.encode() for name in _motif_names(pwms)]
    motif_off = np.zeros(len(mtext) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in mtext], out=motif_off[1:])
    single = np.zeros(max(len(pwms), 1), dtype=np.int64)
    single[table.a] = table.n_a
    single[table.b] = table.n_b
    n = len(order)

    def col(x, dtype, ct):
        if x is None or n == 0:
            return None, None
        a = np.ascontiguousarray(np.asarray(x)[order], dtype=dtype)
        return a, _lib.ptr(a, ct)
    cols = [col(table.a, np.int32, ctypes.c_int32), col(table.b, np.int32, ctypes.c_int32)]
    cols += [col(table.n_both, np.int64, ctypes.c_int64)]
    cols += [col(getattr(table, f), np.float64, ctypes.c_double)
             for f in ("expected", "ratio", "p_cooccur", "p_exclusive", "q_cooccur")]
    cols += [col(table.n_both_control, np.int64, ctypes.c_int64)]
    cols += [col(getattr(table, f), np.float64, ctypes.c_double)
             for f in ("fold_change", "p_enriched", "p_depleted", "p_corrected")]
    ptrs = [c[1] for c in cols]
    _lib.check(lib.msb_write_cooccur_table(
        os.path.join(output_dir, "motif_cooccurrence.xls").encode(), COOCCUR_HEADER.encode(), n, ptrs[0], ptrs[1], len(pwms),
        b"".join(mtext), _lib.ptr(motif_off, ctypes.c_int64), _lib.ptr(single, ctypes.c_int64), *ptrs[2:],
        min(os.cpu_count() or 1, 32)))


def write_spacing_table(output_dir, pwms, anchors, rows):
    """motif_spacing.xls: one row per (anchor, partner, orientation) with at least one pair (cooccur.spacing_rows):
    the pairs at all offsets, the peak offset among the non-overlapping ones and its pairs, the pairs expected per
    such offset, the peak's p-value (`NA` when every offset overlaps) and the counts from -D to D."""
    os.makedirs(output_dir, exist_ok=True)
    names = _motif_names(pwms)

    def na(v):
        return "NA" if v is None or (isinstance(v, float) and np.isnan(v)) else str(v)
    with open(os.path.join(output_dir, "motif_spacing.xls"), "w") as out:
        out.write(SPACING_HEADER)
        for r in rows:
            out.write(f"{names[anchors[r.anchor]]}\t{names[r.partner]}\t{'same' if r.orientation == 0 else 'opposite'}\t"
                      f"{r.pairs}\t{na(r.peak_offset)}\t{na(r.peak_pairs)}\t{na(r.expected)}\t{na(r.p_value)}\t"
                      f"{','.join(map(str, r.counts.tolist()))}\n")


CENTRALITY_HEADER = ("Motif_ID\tMotif_name\tLength\tTested_regions\tRegions_with_site\tHalf_width\tCentral_best_sites\t"
                     "Expected\tRatio\tP_value\tCorrected_P_value\n")


def write_centrality_tables(output_dir, pwms, result, rows):
    """motif_centrality.xls: one row per motif (centrality.centrality_rows, in its order), `NA` where the motif has no
    site in a tested region or no width to test; motif_site_distribution.xls: per motif a row of all its sites and a row
    of the regions' best sites, one column per bin headed by the bin centre k B (bases from the summit)."""
    os.makedirs(output_dir, exist_ok=True)

    def na(v):
        return "NA" if v is None or (isinstance(v, float) and np.isnan(v)) else str(v)
    with open(os.path.join(output_dir, "motif_centrality.xls"), "w") as out:
        out.write(CENTRALITY_HEADER)
        for r in rows:
            p = pwms[r.motif]
            out.write(f"{p.matrix_id}\t{p.name}\t{r.length}\t{r.n_tested}\t{r.n_regions}\t{na(r.half_width)}\t"
                      f"{na(r.central)}\t{na(r.expected)}\t{na(r.ratio)}\t{na(r.p_value)}\t{na(r.p_corrected)}\n")
    K = (result.hist_all.shape[1] - 1) // 2
    with open(os.path.join(output_dir, "motif_site_distribution.xls"), "w") as out:
        out.write("Motif_ID\tMotif_name\tSites\t" + "\t".join(str(k * int(result.bin)) for k in range(-K, K + 1)) + "\n")
        for m, p in enumerate(pwms):
            for what, hist in (("all", result.hist_all), ("best", result.hist_best)):
                out.write(f"{p.matrix_id}\t{p.name}\t{what}\t" + "\t".join(map(str, hist[m].tolist())) + "\n")
