"""Motif scanner for a list of genomic regions -- the reference's `motifscan.scanner` API
(scanner.py:16-193) over the CUDA path.

Same constructor arguments, attributes (`sequences`, `seq_starts`, `seq_ends`) and
`scan_motifs(pwms)` contract; the result indexes like the reference's nested list
`[pwm][region] -> [MotifSite(start, score, strand), ...]` but is backed by the arrays the device
returns, so a (motif, region) cell costs nothing until it is looked at (the reference allocates
one Python list per cell, scanner.py:140-143 -- 3.8e8 lists for configs[4]).
"""
import contextlib
import logging
import os
from collections import namedtuple

import numpy as np

from . import engine
from .centrality import CentralityResult, half_bins
from .cooccur import PairResult

logger = logging.getLogger(__name__)

MotifSite = namedtuple("MotifSite", ["start", "score", "strand"])  # scanner.py:16
_STRAND_ARG = {"+": 1, "-": 2, "both": 3}  # scanner.py:118-123


class _MergedResult:
    """The gathered arrays of several devices' ScanResults, shaped like one (what MotifSites reads)."""

    def __init__(self, results, block_starts, n_motifs, n_seqs):
        counts = np.stack([r.counts for r in results]) if results else np.zeros((0, n_motifs), dtype=np.int64)
        self.counts = counts.sum(axis=0) if len(results) else np.zeros(n_motifs, dtype=np.int64)
        self.offsets = np.zeros(n_motifs + 1, dtype=np.int64)
        np.cumsum(self.counts, out=self.offsets[1:])
        self.n_sites = int(self.counts.sum())
        # per motif: device 0's sites, then device 1's, ... -- the devices hold ascending blocks of regions,
        # so this is the reference's (motif, region, start) order; region indices become global on the way
        groups = [np.arange(a, b, dtype=np.int32) for a, b in zip(block_starts, list(block_starts[1:]) + [n_seqs])]
        self.seq_idx, self.start, self.score, self.strand = engine.merge_sites(
            counts, [r.seq_idx for r in results], [r.start for r in results], [r.score for r in results],
            [r.strand for r in results], seq_to_group=groups)
        for r in results:
            r.close()


class Scanner:
    def __init__(self, genome, regions, window_size=0, strand="both", p_value="1e-4",
                 remove_dup=True, n_threads=1, device=None, devices=None):
        self.window_size = window_size if window_size > 0 else 0
        self.extend = window_size // 2
        if strand not in _STRAND_ARG:
            raise ValueError(f"invalid strand option: {strand!r}")
        self.strand = strand
        self.p_value = p_value
        self.remove_dup = remove_dup
        # kept for signature compatibility (scanner.py:56-66); the GPU path has no thread count
        self.n_threads = max(1, min(int(n_threads), os.cpu_count() or 1))
        self.device = device
        # several GPUs of this process: the regions are dealt to them in contiguous blocks, one host thread
        # and one context per GPU (the reference's n_threads pool over motifs, cscore.c:323-328, 425-436)
        self.devices = list(devices) if devices is not None else None
        self.seq_starts = []
        self.seq_ends = []
        self._chunks = []
        self._chroms = []
        self._sequences = None
        # a genome.DeviceGenome keeps the packed chromosomes in HBM: windows are cut out on the device;
        # a genome.PackedGenome (host planes) is made resident on every device that scans
        self._resident = genome if hasattr(genome, "extract") and hasattr(genome, "chrom_index") else None
        self._packed = genome if self._resident is None and hasattr(genome, "planes") else None
        self._genome = genome
        self._extract_seq(genome, regions)

    def _extract_seq(self, genome, regions):
        """Forward-strand sequence of every region's scan window (scanner.py:71-87): the whole
        region, or `window_size` centred on the summit, clipped to [0, chromosome size)."""
        fetch = getattr(genome, "fetch_bytes", None)
        sizes = genome.chrom_sizes
        for region in regions:
            if self.window_size <= 0:
                start, end = region.start, region.end
            else:
                start = max(region.summit - self.extend, 0)
                end = min(region.summit + self.extend, sizes[region.chrom])
            self.seq_starts.append(start)
            self.seq_ends.append(end)
            if self._resident is not None or self._packed is not None:
                genome.chrom_index[region.chrom]   # KeyError for unknown chromosomes, as fetch raises
                self._chroms.append(region.chrom)
            elif fetch is not None:
                self._chunks.append(fetch(region.chrom, start, end))
            else:
                self._chunks.append(genome.fetch_sequence(region.chrom, start, end).encode("utf-8"))

    @property
    def sequences(self):
        if self._sequences is None:
            if self._resident is not None or self._packed is not None:   # only materialised when somebody asks for the strings
                self._sequences = [self._genome.fetch_sequence(c, a, b)
                                   for c, a, b in zip(self._chroms, self.seq_starts, self.seq_ends)]
            else:
                self._sequences = [c.decode("utf-8") for c in self._chunks]
        return self._sequences

    def scan_motifs(self, pwms, ctx=None, pairs=None, centrality=None):
        """Scan for motif occurrences; returns a `MotifSites` (nested-list view, (n_pwms,
        n_regions, n_sites)).  `pairs` (a cooccur.PairSpec): also reduce the final sites on the device to motif pair
        counts and / or anchor spacing histograms, summed over the devices' blocks, as `MotifSites.pairs`.
        `centrality` (a bin width B, 1 <= B <= window_size // 2): also reduce them to the histograms of the sites'
        offsets from the summits in the windows that no chromosome end clips, summed likewise, as
        `MotifSites.centrality` (a centrality.CentralityResult)."""
        cutoffs = []
        for pwm in pwms:
            try:
                cutoffs.append(pwm.cutoffs[self.p_value])
            except (TypeError, KeyError):
                raise ValueError(f"PWM has no motif score cutoff set for P-value {self.p_value!r}")
        matrices = [pwm.matrix for pwm in pwms]
        lengths = [pwm.length for pwm in pwms]
        if pairs is not None and pairs.anchors and not all(0 <= int(a) < len(matrices) for a in pairs.anchors):
            raise ValueError("spacing anchor index out of range")
        mid2 = None
        if centrality is not None:
            E, B = self.extend, int(centrality)
            if self.window_size == 0 or E < 1:
                raise ValueError("centrality needs summit-centred windows (window_size >= 2)")
            if not 1 <= B <= E:
                raise ValueError(f"centrality bin width must be 1..{E} (window_size // 2), got {B}")
            K = half_bins(E, B)
            # twice the summit's offset in its window, or -1 for a window a chromosome end clipped
            mid2 = np.where(np.asarray(self.seq_ends, dtype=np.int64) - np.asarray(self.seq_starts, dtype=np.int64) == 2 * E,
                            2 * E, -1).astype(np.int32)
            n_tested = int((mid2 >= 0).sum())
            if n_tested < len(mid2):
                logger.info(f"Centrality: {len(mid2) - n_tested} of {len(mid2)} regions have windows clipped by a "
                            "chromosome end and are left out")
        if not matrices:
            sites = MotifSites(None, 0, self.seq_starts, lengths)
            if pairs is not None:
                sites.pairs = PairResult(np.zeros((0, 0), dtype=np.int64) if pairs.cooccur else None, len(self.seq_starts), None)
            if centrality is not None:
                empty = np.zeros((0, 2 * K + 1), dtype=np.int64)
                sites.centrality = CentralityResult(empty, empty.copy(), n_tested, E, B)
            return sites
        if self._resident is not None:
            ctxs = [self._resident.ctx]       # the windows live where the genome lives
        elif ctx is not None:
            ctxs = [ctx]
        elif self.devices:
            ctxs = [engine.default_context(d) for d in self.devices]
        else:
            dev = self.device
            if dev is None:
                dev = int(os.environ.get("MOTIFSCAN_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
            ctxs = [engine.default_context(dev)]
        n = len(self.seq_starts)
        ctxs = ctxs[:max(1, min(len(ctxs), n))]
        bounds = [n * k // len(ctxs) for k in range(len(ctxs) + 1)]    # contiguous blocks of regions
        strand = _STRAND_ARG[self.strand]

        def reduce_pairs(c, motifs, n_block):
            """The pair reductions of the scan just run on `c` (the caller holds c._lock)."""
            counts = c.pair_counts(len(matrices), n_block) if pairs.cooccur else None
            hist = c.spacing(motifs, list(pairs.anchors), pairs.max_offset) if pairs.anchors else None
            return counts, hist

        def reduce_block(c, motifs, a, b):
            """The reductions of the scan of regions a..b just run on `c` (the caller holds c._lock)."""
            return (reduce_pairs(c, motifs, b - a) if pairs is not None else None,
                    c.centrality(motifs, mid2[a:b], B, K) if centrality is not None else None)

        def scan_block(k):
            c, a, b = ctxs[k], bounds[k], bounds[k + 1]
            motifs = engine.MotifSet(c, matrices, cutoffs)
            try:
                # the reductions read the scan's sites on the device: no other scan on a shared context may come between
                with c._lock if pairs is not None or centrality is not None else contextlib.nullcontext():
                    if self._resident is not None or self._packed is not None:
                        dg = self._resident if self._resident is not None else self._packed_on(c)
                        sset = dg.extract(self._chroms[a:b], self.seq_starts[a:b], self.seq_ends[a:b])
                        try:
                            res = engine.scan(c, motifs, sset, strand, remove_dup=self.remove_dup)
                        finally:
                            sset.close()
                    else:
                        chunks = self._chunks[a:b]
                        off = np.zeros(len(chunks) + 1, dtype=np.int64)
                        if chunks:
                            np.cumsum([len(x) for x in chunks], out=off[1:])
                        blob = np.frombuffer(b"".join(chunks), dtype=np.uint8)
                        res = engine.scan_ascii(c, motifs, blob, off, strand, remove_dup=self.remove_dup)
                    if pairs is None and centrality is None:
                        return res, None
                    return res, reduce_block(c, motifs, a, b)
            finally:
                motifs.close()

        if len(ctxs) == 1:
            res, reduced = scan_block(0)
            res = res.detach()
            blocks = [reduced]
        else:
            import concurrent.futures
            with concurrent.futures.ThreadPoolExecutor(max_workers=len(ctxs)) as pool:
                out = list(pool.map(scan_block, range(len(ctxs))))
            res = _MergedResult([r for r, _ in out], bounds[:-1], len(matrices), n)
            blocks = [p for _, p in out]
        sites = MotifSites(res, len(matrices), self.seq_starts, lengths)
        # the blocks hold disjoint regions: their counts and histograms add up
        if pairs is not None:
            counts = sum(p[0][0] for p in blocks) if pairs.cooccur else None
            hist = sum(p[0][1] for p in blocks) if pairs.anchors else None
            sites.pairs = PairResult(counts, n, hist)
        if centrality is not None:
            sites.centrality = CentralityResult(sum(p[1][0] for p in blocks), sum(p[1][1] for p in blocks), n_tested, E, B)
        return sites

    def _packed_on(self, ctx):
        """The device-resident copy of a host PackedGenome on `ctx`'s GPU (made on first use, kept on the
        PackedGenome so that target and control scanners share it)."""
        from .genome import DeviceGenome
        cache = self._packed.__dict__.setdefault("_device_copies", {})
        if ctx.device not in cache:
            cache[ctx.device] = DeviceGenome(self._packed, ctx)
        return cache[ctx.device]


class _PerMotif:
    """`motif_sites[m]`: sequence-indexed view of one motif's sites."""

    def __init__(self, parent, m):
        self._p = parent
        self._m = m
        a, b = parent._off[m], parent._off[m + 1]
        self._a = a
        seq = parent._seq_idx[a:b]
        # sites are sorted by sequence within a motif: CSR over sequences by binary search
        self._bounds = a + np.searchsorted(seq, np.arange(parent.n_seqs + 1))

    def __len__(self):
        return self._p.n_seqs

    def __getitem__(self, s):
        if isinstance(s, slice):
            return [self[i] for i in range(*s.indices(len(self)))]
        if s < 0:
            s += len(self)
        if not 0 <= s < len(self):
            raise IndexError("region index out of range")
        p = self._p
        a, b = int(self._bounds[s]), int(self._bounds[s + 1])
        base = p.seq_starts[s]
        return [MotifSite(start=base + int(p._start[k]), score=float(p._score[k]),
                          strand="+" if p._strand[k] == 1 else "-") for k in range(a, b)]

    def __iter__(self):
        return (self[s] for s in range(len(self)))

    def site_counts(self):
        """Number of sites per region (what motif_sites_number.xls tabulates, io/__init__.py:27)."""
        return np.diff(self._bounds)


class MotifSites:
    """Nested-list view `[pwm][region] -> [MotifSite]` over the scan's arrays (the shape
    make_motif_sites returns, scanner.py:135-153).  `start` is genomic: window start + offset."""

    def __init__(self, res, n_pwms, seq_starts, lengths):
        self.n_pwms = n_pwms
        self.n_seqs = len(seq_starts)
        self.seq_starts = list(seq_starts)
        self.lengths = list(lengths)
        self.pairs = None    # cooccur.PairResult when the scan was asked for pair reductions
        self.centrality = None    # centrality.CentralityResult when the scan was asked for the positional histograms
        if res is None:
            self._off = np.zeros(n_pwms + 1, dtype=np.int64)
            self._seq_idx = np.zeros(0, dtype=np.int32)
            self._start = np.zeros(0, dtype=np.int32)
            self._score = np.zeros(0, dtype=np.float64)
            self._strand = np.zeros(0, dtype=np.int8)
        else:
            self._off, self._seq_idx = res.offsets, res.seq_idx
            self._start, self._score, self._strand = res.start, res.score, res.strand

    def __len__(self):
        return self.n_pwms

    def __getitem__(self, m):
        if isinstance(m, slice):
            return [self[i] for i in range(*m.indices(len(self)))]
        if m < 0:
            m += len(self)
        if not 0 <= m < len(self):
            raise IndexError("motif index out of range")
        return _PerMotif(self, m)

    def __iter__(self):
        return (self[m] for m in range(len(self)))

    def tolist(self):
        return [[cell for cell in per] for per in self]

    # -- vectorised summaries (consumers: stats.motif_enrichment, the site tables) --------------
    def n_sites(self):
        return np.diff(self._off)

    def regions_with_sites(self):
        """Per motif, the number of regions with at least one site (stats.py:29-31)."""
        out = np.zeros(self.n_pwms, dtype=np.int64)
        seq = self._seq_idx
        if len(seq) == 0:
            return out
        # a site opens a new (motif, region) cell if it is the first of its motif or its region differs
        # from the previous site's; cells per motif = segment sums (sites are sorted by motif, region)
        first = np.empty(len(seq), dtype=bool)
        first[0] = True
        np.not_equal(seq[1:], seq[:-1], out=first[1:])
        nonempty = np.flatnonzero(np.diff(self._off) > 0)
        starts = np.asarray(self._off)[nonempty]
        first[starts] = True
        out[nonempty] = np.add.reduceat(first, starts, dtype=np.int64)
        return out


# ---- list-based helpers with the reference's signatures (scanner.py:135-193) ---------------------
def make_motif_sites(sites, seq_starts):
    """Pooled `c_scan_motif` output -> nested list (n_pwms, n_seqs, n_sites) with genomic starts
    and '+'/'-' strands (scanner.py:135-153)."""
    nested = []
    for per_pwm in sites:
        cells = [[] for _ in seq_starts]
        for seq_idx, pos, score, strand in per_pwm:
            cells[seq_idx].append(MotifSite(seq_starts[seq_idx] + pos, score, "+" if strand == 1 else "-"))
        nested.append(cells)
    return nested


def _survivors(sites, length):
    """One strand's sites by ascending start -> survivors of the reference's greedy pass
    (scanner.py:156-168): a site closer than `length` to the current survivor replaces it only
    when it scores strictly higher."""
    kept = []
    for site in sites:
        if kept and site.start - kept[-1].start < length:
            if kept[-1].score >= site.score:
                continue
            kept.pop()
        kept.append(site)
    return kept


def deduplicate_motif_sites(motif_sites, lengths):
    """Adjacent-site de-duplication (scanner.py:171-193), per strand, then merged by start with
    '+' first on ties (the reference's stable sort of fwd + rev)."""
    out = []
    for per_pwm, length in zip(motif_sites, lengths):
        cells = []
        for sites in per_pwm:
            fwd = _survivors([s for s in sites if s.strand == "+"], length)
            rev = _survivors([s for s in sites if s.strand != "+"], length)
            cells.append(sorted(fwd + rev, key=lambda s: s.start))
        out.append(cells)
    return out
