"""`motifscan scan` and `motifscan motif --build` over the CUDA scan path.

Same flags as the reference's subcommands (cli/main.py:407-430, 504-579) and the same outputs
(cli/scan.py:24-108, cli/motif.py:101-155).  Differences, all outside the scan path:
  * `-g` / `-m` are resolved through `~/.motifscanrc` ([genome] / [motif] sections, the
    reference's registry format, config.py:15-117) or taken as a directory path when one exists;
  * `--loc`, `--plot` and the install / list / search subcommands (gene annotation, matplotlib,
    remote databases) are out of scope (SURVEY.md section 2 rows 7-9, 13) and exit with a message;
  * `-t` is accepted and ignored: the device has no thread count; `--gpus N` scans on the first N
    GPUs of the box (one host thread and one context per GPU, results gathered in region order);
  * control regions are always whole-background random (`generate_control_regions` without genes):
    the gene-distance-matched branch of cli/scan.py needs the annotation layer, which is out of
    scope -- when the genome directory holds an annotation file a warning says so;

  * `scan --whole-genome` (instead of `-i`) scans every chromosome end to end and writes exactly what
    `scan -i <one BED line "chrom 0 size" per chromosome> -w 0 --no-enrich` writes: one table row per
    chromosome and, with `--site`, the de-duplicated sites.  The genome is always scanned through its packed
    planes (`<name>.packed.*` cache, written when missing), cut into equal-work shares with `--gpus N`;
    de-duplication runs per piece on the device and the chains of overlapping sites that cross a piece
    boundary are joined on the host.  There is no control set, so no enrichment: `-c`, `--cf` and `--loc` are
    errors; `-w`, `--n-random` and `--seed` are ignored;

  * `variant` (not in the reference) scans the SNVs and MNVs of a VCF against the resident genome and reports the
    motif sites each allele creates or destroys (motifscan_b200/variants.py; one GPU, `-t` ignored); `--indels` scans
    insertions and deletions too, as the VCF places them (normalise it first); `--haplotypes` reads the phased
    genotypes and scans the alleles each haplotype carries within a motif width of each other together;

  * `scan --cooccur` (not in the reference) also writes motif_cooccurrence.xls: for every motif pair, the regions with
    sites of both, tested for co-occurrence and mutual exclusion within the input and, unless --no-enrich, against the
    control regions; `scan --spacing-anchor ID[,ID...] [--spacing-max D]` writes motif_spacing.xls: per anchor motif,
    partner motif and orientation, the partner sites at offsets -D..D of the anchor's sites (default D = 50) and the
    most enriched non-overlapping offset (motifscan_b200/cooccur.py).  Both are errors with --whole-genome;

  * `scan --centrality [--centrality-bin B]` (not in the reference) writes where each motif's sites fall around the
    region summits: motif_site_distribution.xls, per motif the sites and the best site of each region in bins of B bases
    (default 10) by their centre's offset from the summit, and motif_centrality.xls, a test of the best sites piling up
    within +-(j + 1/2) B of the summit against a uniform position, at the most significant width
    (motifscan_b200/centrality.py).  Only windows that no chromosome end clips are used; the control regions are not
    (a random window has no summit).  An error with --whole-genome and with -w below 2;

    python -m motifscan_b200 scan -i peaks.bed -m <motif set> -g <genome> -o out_dir
    python -m motifscan_b200 scan -i peaks.bed -m <motif set> -g <genome> -o out_dir --cooccur --spacing-anchor MA0099.3
    python -m motifscan_b200 scan -i peaks.narrowPeak -f narrowpeak -m <motif set> -g <genome> -o out_dir --centrality
    python -m motifscan_b200 scan --whole-genome -m <motif set> -g <genome> -o out_dir [--site]
    python -m motifscan_b200 motif --build <motif set> -g <genome>
    python -m motifscan_b200 variant -i calls.vcf.gz -m <motif set> -g <genome> -o out_dir [--indels]
    python -m motifscan_b200 variant -i phased.vcf.gz -m <motif set> -g <genome> -o out_dir --haplotypes [--samples A,B]
"""
import argparse
import logging
import os
import sys
from configparser import ConfigParser

from . import io as msio
from .builder import build_cutoffs
from .centrality import centrality_rows
from .cooccur import PairSpec, cooccur_table, spacing_rows
from .genome import Genome
from .motif import MotifPwms, PositionWeightMatrix, pfm_to_pwm, read_jaspar_pfms
from .region import REGION_FORMATS, generate_control_regions, load_motifscan_regions
from .scanner import Scanner
from .stats import motif_enrichment

logger = logging.getLogger("motifscan")
RC_PATH = os.path.expanduser("~/.motifscanrc")


def _registry(section, name, rc_path=None):
    """Directory registered for `name` in the reference's rc file, or `name` itself if it is one."""
    if os.path.isdir(name):
        return os.path.abspath(name), os.path.basename(os.path.normpath(name))
    cfg = ConfigParser()
    cfg.read(rc_path or os.environ.get("MOTIFSCANRC", RC_PATH))
    if cfg.has_option(section, name):
        return cfg.get(section, name), name
    raise SystemExit(f"motifscan: error: {section} {name!r} not found (not a directory, not in the rc file)")


def load_genome(name):
    path, short = _registry("genome", name)
    return Genome(short, path=path)


PACKED_MIN_BP = 1 << 26    # scans of at least this many window bases go through the packed, device-resident genome
BUILD_RESIDENT_MIN_SAMPLES = 200000    # `motif --build` with at least this many background samples samples from it too


def packed_genome(genome, window_bp, device=0):
    """The genome's packed planes (`genome.PackedGenome`, 0.375 B/bp) for a scan of `window_bp` bases, or None to
    fetch region strings from the FASTA as the reference does (scanner.py:76-87).  A cache written next to the
    FASTA (`<name>.packed.*`, like the `.fai`) is always used; without one the genome is encoded on the GPU and
    the cache written when the scan is large enough to pay for it (one pass over the FASTA)."""
    from . import engine
    from .genome import PackedGenome
    prefix = os.path.join(genome.path, f"{genome.name}.packed") if genome.path else None
    if prefix and os.path.isfile(prefix + ".chroms.tsv"):
        try:
            pg = PackedGenome.load(prefix, genome=genome)
            if pg.chrom_sizes == genome.chrom_sizes:
                return pg
            logger.warning("packed genome cache does not match the FASTA index: ignored")
        except (OSError, ValueError) as err:
            logger.warning(f"packed genome cache unreadable ({err}): ignored")
    if window_bp < PACKED_MIN_BP:
        return None
    logger.info("Packing the genome (2 bits per base + N mask) on the device")
    pg = PackedGenome.from_genome(genome, engine.default_context(device))
    if prefix:
        try:
            pg.save(prefix)
        except OSError:
            pass
    return pg


def pwms_path(motif_dir, name, genome_name):
    return os.path.join(motif_dir, f"{name}_{genome_name}_pwms.motifscan")   # motif/__init__.py:22


def load_built_pwms(name, genome_name):
    motif_dir, short = _registry("motif", name)
    path = pwms_path(motif_dir, short, genome_name)
    if not os.path.isfile(path):
        raise SystemExit(f"motifscan: error: PWMs of motif set {short!r} are not built for genome "
                         f"{genome_name!r} (run: motif --build {name} -g {genome_name})")
    pwms = MotifPwms(name=short, genome=genome_name)
    pwms.read_motifscan_pwms(path)
    return pwms


def run_whole_genome(args):
    """`scan --whole-genome`: every chromosome as one region, through GenomeScanner with remove_dup."""
    import time
    from .genome_scan import GenomeScanner
    from .region import GenomicRegion
    logger.info("===== Loading data =====")
    genome = load_genome(args.genome)
    pwms = load_built_pwms(args.motif, genome.name)
    try:
        cutoffs = [pwm.cutoffs[args.p_value] for pwm in pwms]
    except (TypeError, KeyError):
        raise SystemExit(f"motifscan: error: PWMs have no motif score cutoff set for P-value {args.p_value!r}")
    logger.info("===== Scanning motifs (whole genome) =====")
    devices = _devices(args.n_gpus)
    pg = packed_genome(genome, PACKED_MIN_BP, devices[0])
    regions = [GenomicRegion(c, 0, genome.chrom_sizes[c]) for c in pg.chroms]
    t0 = time.perf_counter()
    gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, strand=args.strand, devices=devices, remove_dup=True)
    try:
        sites = gs.scan(collect_sites=args.report_site)
    finally:
        gs.close()
    seconds = time.perf_counter() - t0
    total_bp = sum(genome.chrom_sizes[c] for c in pg.chroms)
    logger.info(f"Scanned {len(pwms)} motifs x {total_bp} bp in {seconds:.3f} s: "
                f"{len(pwms) * total_bp / max(seconds, 1e-12):.3e} motif*bp/s, {int(sites.counts.sum())} sites")
    logger.info("Saving the result tables")
    msio.write_cell_tables(args.output_dir, pwms, regions, sites.cell_counts.T, sites.cell_best.T)
    if args.report_site:
        msio.write_sites_bed(args.output_dir, pwms, regions, sites)
    logger.info("===== MotifScan Finished =====")
    return 0


def run_scan(args):
    if args.whole_genome == (args.input_file is not None):
        raise SystemExit("motifscan scan: error: give exactly one of -i and --whole-genome")
    if args.whole_genome:
        for flag, given in (("-c", args.control_file is not None), ("--cf", args.control_format_given),
                            ("--loc", args.location is not None), ("--cooccur", args.cooccur),
                            ("--spacing-anchor", args.spacing_anchor is not None)):
            if given:
                raise SystemExit(f"motifscan scan: error: {flag} has no meaning with --whole-genome (no enrichment, and a "
                                 "chromosome is not a region to co-occur in)")
        if args.centrality:
            raise SystemExit("motifscan scan: error: --centrality has no meaning with --whole-genome (a chromosome has no "
                             "summit to be central to)")
        if args.plot_dist:
            raise SystemExit("motifscan scan: --plot needs matplotlib, which is out of scope here")
        return run_whole_genome(args)
    if args.location is not None:
        raise SystemExit("motifscan scan: --loc needs the gene annotation layer, which is out of scope here")
    if args.plot_dist:
        raise SystemExit("motifscan scan: --plot needs matplotlib, which is out of scope here")
    if args.centrality:
        extend = args.window_size // 2
        if extend < 1:
            raise SystemExit("motifscan scan: error: --centrality needs windows centred on the summits (-w 2 or more): "
                             "regions of their own lengths share no geometry to test positions against")
        if args.centrality_bin > extend:
            raise SystemExit(f"motifscan scan: error: --centrality-bin must be 1..{extend} (half of -w), "
                             f"got {args.centrality_bin}")
    logger.info("===== Loading data =====")
    genome = load_genome(args.genome)
    pwms = load_built_pwms(args.motif, genome.name)
    anchors = resolve_anchors(pwms, args.spacing_anchor) if args.spacing_anchor is not None else []
    pairs = None
    if args.cooccur or anchors:
        pairs = PairSpec(cooccur=args.cooccur, anchors=anchors, max_offset=args.spacing_max)
    regions = load_motifscan_regions(args.input_file, args.input_format)
    logger.info("===== Scanning motifs =====")
    devices = _devices(args.n_gpus)
    window_bp = sum((args.window_size if args.window_size > 0 else r.end - r.start) for r in regions)
    source = packed_genome(genome, window_bp * (1 if args.no_enrich else 2), devices[0]) or genome
    common = dict(genome=source, window_size=args.window_size, strand=args.strand, p_value=args.p_value,
                  remove_dup=True, n_threads=args.n_threads, devices=devices)
    sites = Scanner(regions=regions, **common).scan_motifs(pwms, pairs=pairs,
                                                          centrality=args.centrality_bin if args.centrality else None)
    logger.info("Saving the result tables")
    msio.write_sites_table(args.output_dir, pwms, regions, sites)
    if args.report_site:
        msio.write_sites_bed(args.output_dir, pwms, regions, sites)
    if anchors:
        rows = spacing_rows(sites.pairs.spacing, anchors, [int(p.length) for p in pwms])
        msio.write_spacing_table(args.output_dir, pwms, anchors, rows)
    if args.centrality:
        import time
        t0 = time.perf_counter()
        rows = centrality_rows(sites.centrality, [int(p.length) for p in pwms])
        t1 = time.perf_counter()
        msio.write_centrality_tables(args.output_dir, pwms, sites.centrality, rows)
        logger.info(f"Centrality of {len(pwms)} motifs in {sites.centrality.n_tested} of {len(regions)} regions: "
                    f"statistics {t1 - t0:.3f} s, tables {time.perf_counter() - t1:.3f} s")
    control_pairs = None
    if not args.no_enrich:
        logger.info("===== Motif Enrichment =====")
        if args.control_file:
            controls = load_motifscan_regions(args.control_file, args.control_format)
        else:
            if genome.path and any(f.endswith(("_gene_annotation.txt", "refGene.txt")) for f in os.listdir(genome.path)):
                logger.warning("gene annotation found but unused: control regions are drawn from the whole "
                               "background, not matched by gene distance as the reference does (out of scope)")
            controls = generate_control_regions(args.n_random, regions, genome.chrom_sizes, random_seed=args.seed)
        control_sites = Scanner(regions=controls, **common).scan_motifs(
            pwms, pairs=PairSpec(cooccur=True) if args.cooccur else None)
        msio.write_enrich_table(args.output_dir, motif_enrichment(pwms, sites, control_sites))
        control_pairs = control_sites.pairs
    if args.cooccur:
        import time
        logger.info("===== Motif Co-occurrence =====")
        t0 = time.perf_counter()
        table = cooccur_table(sites.pairs.counts, sites.pairs.n_regions,
                              control_pairs.counts if control_pairs else None,
                              control_pairs.n_regions if control_pairs else None, n_threads=COOCCUR_THREADS)
        t1 = time.perf_counter()
        msio.write_cooccur_table(args.output_dir, pwms, table)
        logger.info(f"Co-occurrence of {len(table.a)} motif pairs: statistics {t1 - t0:.3f} s, "
                    f"table {time.perf_counter() - t1:.3f} s")
    logger.info("===== MotifScan Finished =====")
    return 0


def run_variant(args):
    """`variant`: sites gained / lost by the SNVs and MNVs (and with --indels the indels) of a VCF
    (variants.read_vcf / scan_variants)."""
    from . import variants as msvar
    from .genome import DeviceGenome
    logger.info("===== Loading data =====")
    genome = load_genome(args.genome)
    pwms = load_built_pwms(args.motif, genome.name)
    try:
        cutoffs = [pwm.cutoffs[args.p_value] for pwm in pwms]
    except (TypeError, KeyError):
        raise SystemExit(f"motifscan: error: PWMs have no motif score cutoff set for P-value {args.p_value!r}")
    if args.samples and not args.haplotypes:
        raise SystemExit("motifscan variant: error: --samples needs --haplotypes")
    samples = None
    if args.haplotypes:
        samples = [x for x in args.samples.split(",") if x] if args.samples else "all"
    pg = packed_genome(genome, PACKED_MIN_BP)
    try:
        vcf = msvar.read_vcf(args.input_file, pg, indels=args.indels, samples=samples)
    except (OSError, UnicodeDecodeError, EOFError) as err:
        raise SystemExit(f"motifscan variant: error: cannot read {args.input_file}: {err}")
    except ValueError as err:
        raise SystemExit(f"motifscan variant: error: {err}")
    if args.haplotypes:
        return _run_haplotypes(args, msvar, pg, pwms, cutoffs, vcf)
    logger.info("===== Scanning variants =====")
    dg = DeviceGenome(pg)
    try:
        sites = msvar.scan_variants(dg, pwms, cutoffs, vcf, strand=args.strand)
    finally:
        dg.close()
    by = sites.rows_by_effect()
    skipped = ", ".join(f"{k} {v}" for k, v in vcf.skipped.items())
    n_indels = f", {sum(len(r) != len(a) for r, a in zip(vcf.ref, vcf.alt))} of them indels" if args.indels else ""
    logger.info(f"Scanned {len(vcf)} alleles{n_indels} (skipped: {skipped}) x {len(pwms)} motifs, {sites.motif_bp:.3e} motif*bp "
                f"in {sites.seconds:.3f} s: {len(sites)} rows ({by['gain']} gain, {by['loss']} loss, {by['both']} both)")
    logger.info("Saving the result tables")
    msio.write_variant_tables(args.output_dir, pwms, vcf, sites)
    logger.info("===== MotifScan Finished =====")
    return 0


def _run_haplotypes(args, msvar, pg, pwms, cutoffs, vcf):
    """`variant --haplotypes`: sites gained / lost by each phased haplotype's clusters of alleles
    (variants.haplotype_clusters / scan_haplotypes)."""
    from .genome import DeviceGenome
    lmax = max((int(p.length) for p in pwms), default=1)
    haps = msvar.haplotype_clusters(vcf, lmax)
    skipped = ", ".join(f"{k} {v}" for k, v in vcf.skipped.items())
    calls = ", ".join(f"{k} {v}" for k, v in {**vcf.call_skipped, "overlap": haps.overlap}.items())
    logger.info(f"Read {len(vcf)} alleles (skipped: {skipped}) and {len(vcf.call_allele)} haplotype calls of "
                f"{len(vcf.samples)} samples (skipped: {calls}): {len(haps)} distinct clusters")
    logger.info("===== Scanning haplotypes =====")
    dg = DeviceGenome(pg)
    try:
        sites = msvar.scan_haplotypes(dg, pwms, cutoffs, haps, strand=args.strand)
    finally:
        dg.close()
    by = sites.rows_by_effect()
    logger.info(f"Scanned {len(haps)} clusters x {len(pwms)} motifs, {sites.motif_bp:.3e} motif*bp in {sites.seconds:.3f} s: "
                f"{len(sites)} rows ({by['gain']} gain, {by['loss']} loss, {by['both']} both)")
    logger.info("Saving the result tables")
    msio.write_haplotype_tables(args.output_dir, pwms, haps, sites)
    logger.info("===== MotifScan Finished =====")
    return 0


def run_motif(args):
    if not args.build:
        raise SystemExit("motifscan motif: only --build is provided here (install / list need the remote databases)")
    if not args.genome:
        raise SystemExit("motifscan motif --build: error: argument -g/--genome is required")
    genome = load_genome(args.genome)
    motif_dir, short = _registry("motif", args.build)
    pfm_path = os.path.join(motif_dir, f"{short}_pfms.jaspar")               # motif/__init__.py:21
    if not os.path.isfile(pfm_path):
        raise SystemExit(f"motifscan motif --build: error: {pfm_path} not found")
    logger.info("Converting motif PFMs to PWMs")
    pwms = MotifPwms(name=short, genome=genome.name)
    for matrix_id, name, pfm in read_jaspar_pfms(pfm_path):
        pwms.append(PositionWeightMatrix(pfm_to_pwm(pfm, genome.bg_freq), name=name, matrix_id=matrix_id))
    logger.info("Sampling background sequences and scoring them on the device")
    # a large sample is drawn from the device-resident genome: the reference's RNG sequence stays on the host, the N
    # count of every attempt and the sampled windows come out of HBM instead of one FASTA fetch per attempt
    source = genome
    if args.n_random * args.n_repeat >= BUILD_RESIDENT_MIN_SAMPLES or os.path.isfile(
            os.path.join(genome.path or "", f"{genome.name}.packed.chroms.tsv")):
        pg = packed_genome(genome, PACKED_MIN_BP)
        if pg is not None:
            from .genome import DeviceGenome
            source = DeviceGenome(pg)
    build_cutoffs(pwms, source, n_random=args.n_random, n_repeat=args.n_repeat, max_n=args.max_n, seed=args.seed)
    pwms.write_motifscan_pwms(pwms_path(motif_dir, short, genome.name))
    logger.info("Successfully built!")
    return 0


COOCCUR_THREADS = min(os.cpu_count() or 1, 16)   # the scipy calls release the GIL: chunks run in parallel


def resolve_anchors(pwms, text):
    """`--spacing-anchor ID[,ID...]` -> motif indices: each item is a matrix_id or a unique motif name."""
    out = []
    for item in (x.strip() for x in text.split(",")):
        if not item:
            continue
        hits = [i for i, p in enumerate(pwms) if p.matrix_id == item]
        if not hits:
            hits = [i for i, p in enumerate(pwms) if p.name == item]
        if len(hits) != 1:
            listed = ", ".join(f"{pwms[i].matrix_id},{pwms[i].name}" for i in hits)
            what = "unknown" if not hits else f"ambiguous (matches {listed})"
            raise SystemExit(f"motifscan scan: error: --spacing-anchor {item!r} is {what}")
        out.append(hits[0])
    if not 1 <= len(out) <= 16:
        raise SystemExit("motifscan scan: error: --spacing-anchor takes 1 to 16 motifs")
    return out


def _devices(n_gpus):
    """`--gpus N`: the first N CUDA devices of this process (the reference's `-t` pool, cli/main.py:427-430,
    565-568, becomes one host thread per GPU); more than there are is an error, not a silent clamp."""
    from . import _lib
    have = _lib.device_count()
    if n_gpus > have:
        raise SystemExit(f"motifscan: error: --gpus {n_gpus} but only {have} CUDA device(s) are visible")
    return list(range(n_gpus))


def _non_negative(text):
    value = int(text)
    if value < 0:
        raise argparse.ArgumentTypeError(f"expect a non-negative integer, got {text!r}")
    return value


def _positive(text):
    value = int(text)
    if value <= 0:
        raise argparse.ArgumentTypeError(f"expect a positive integer, got {text!r}")
    return value


def _spacing_max(text):
    value = int(text)
    if not 0 <= value <= 500:
        raise argparse.ArgumentTypeError(f"expect an integer in 0..500, got {text!r}")
    return value


def make_parser():
    parser = argparse.ArgumentParser(prog="motifscan", description="MotifScan scan path on B200 (motifscan_b200)")
    sub = parser.add_subparsers(dest="command", required=True)

    scan = sub.add_parser("scan", help="Scan input regions to detect motif occurrences.")
    scan.add_argument("-i", dest="input_file", metavar="FILE")
    scan.add_argument("--whole-genome", dest="whole_genome", action="store_true",
                      help="scan every chromosome end to end instead of -i regions (implies --no-enrich; "
                           "-w, --n-random and --seed are ignored)")
    scan.add_argument("-f", dest="input_format", choices=sorted(REGION_FORMATS), default="bed")
    scan.add_argument("-m", "--motif", dest="motif", required=True, metavar="NAME")
    scan.add_argument("-g", "--genome", dest="genome", required=True, metavar="GENOME")
    scan.add_argument("-p", dest="p_value", default="1e-4", choices=["1e-2", "1e-3", "1e-4", "1e-5", "1e-6"])
    scan.add_argument("--loc", dest="location", choices=["promoter", "distal"], default=None)
    scan.add_argument("--upstream", dest="upstream", type=_positive, default=4000)
    scan.add_argument("--downstream", dest="downstream", type=_positive, default=2000)
    scan.add_argument("-w", "--window-size", dest="window_size", type=_non_negative, default=1000)
    scan.add_argument("--strand", dest="strand", choices=["both", "+", "-"], default="both")
    scan.add_argument("--no-enrich", dest="no_enrich", action="store_true")
    scan.add_argument("--n-random", dest="n_random", type=_non_negative, default=5)
    scan.add_argument("--seed", dest="seed", type=int, default=None)
    scan.add_argument("-c", dest="control_file", metavar="FILE")
    scan.add_argument("--cf", dest="control_format", choices=sorted(REGION_FORMATS), default=None)
    scan.add_argument("-t", "--threads", dest="n_threads", type=int, default=1)
    scan.add_argument("--gpus", dest="n_gpus", type=_positive, default=1, metavar="N",
                      help="GPUs of this box to scan on (regions are dealt to them in contiguous blocks)")
    scan.add_argument("-o", "--output-dir", dest="output_dir", required=True, metavar="DIR")
    scan.add_argument("--site", dest="report_site", action="store_true")
    scan.add_argument("--plot", dest="plot_dist", action="store_true")
    scan.add_argument("--cooccur", action="store_true",
                      help="write motif_cooccurrence.xls: regions with sites of both motifs, for every motif pair")
    scan.add_argument("--spacing-anchor", dest="spacing_anchor", default=None, metavar="ID[,ID...]",
                      help="write motif_spacing.xls: offsets of every motif's sites around these motifs' sites "
                           "(matrix_id or unique name, up to 16)")
    scan.add_argument("--spacing-max", dest="spacing_max", type=_spacing_max, default=50, metavar="D",
                      help="largest |offset| of --spacing-anchor, 0..500 (default 50)")
    scan.add_argument("--centrality", action="store_true",
                      help="write motif_centrality.xls and motif_site_distribution.xls: where each motif's sites fall "
                           "around the region summits, and a test of central enrichment")
    scan.add_argument("--centrality-bin", dest="centrality_bin", type=_positive, default=10, metavar="B",
                      help="bin width of --centrality in bases, 1..(-w)/2 (default 10)")
    scan.add_argument("--verbose", action="store_true")
    scan.set_defaults(func=run_scan)

    variant = sub.add_parser("variant", help="Motif sites gained and lost by the SNVs / MNVs (and indels) of a VCF.")
    variant.add_argument("-i", dest="input_file", required=True, metavar="VCF")
    variant.add_argument("-m", "--motif", dest="motif", required=True, metavar="NAME")
    variant.add_argument("-g", "--genome", dest="genome", required=True, metavar="GENOME")
    variant.add_argument("-p", dest="p_value", default="1e-4", choices=["1e-2", "1e-3", "1e-4", "1e-5", "1e-6"])
    variant.add_argument("--strand", dest="strand", choices=["both", "+", "-"], default="both")
    variant.add_argument("-t", "--threads", dest="n_threads", type=int, default=1)
    variant.add_argument("--indels", action="store_true",
                         help="Also scan insertions and deletions (not left-aligned: normalise the VCF first).")
    variant.add_argument("--haplotypes", action="store_true",
                         help="Scan each sample's phased haplotypes: alleles in cis within a motif width are scanned "
                              "together (writes the motif_haplotype_* tables instead).")
    variant.add_argument("--samples", dest="samples", default=None, metavar="A,B,...",
                         help="With --haplotypes: read only these samples (default: all).")
    variant.add_argument("-o", "--output-dir", dest="output_dir", required=True, metavar="DIR")
    variant.add_argument("--verbose", action="store_true")
    variant.set_defaults(func=run_variant)

    motif = sub.add_parser("motif", help="Motif set commands (only --build here).")
    motif.add_argument("--build", dest="build", metavar="NAME")
    motif.add_argument("-g", "--genome", dest="genome", metavar="GENOME")
    motif.add_argument("--n-random", dest="n_random", type=int, default=1000000)
    motif.add_argument("--n-repeat", dest="n_repeat", type=_positive, default=1)
    motif.add_argument("--max-n", dest="max_n", type=int, default=0)
    motif.add_argument("--seed", dest="seed", type=int, default=None)
    motif.add_argument("-t", "--threads", dest="n_threads", type=int, default=1)
    motif.add_argument("--verbose", action="store_true")
    motif.set_defaults(func=run_motif)
    return parser


def main(argv=None):
    args = make_parser().parse_args(argv)
    if args.command == "scan":
        args.control_format_given = args.control_format is not None
        if args.control_format is None:
            args.control_format = "bed"
    logging.basicConfig(stream=sys.stderr, level=logging.DEBUG if args.verbose else logging.INFO,
                        format="%(message)s")
    return args.func(args)


if __name__ == "__main__":
    sys.exit(main())
