"""Genome-wide scan (BASELINE.json configs[3]): every motif on both strands at every position of
every chromosome, chunked and sharded over the GPUs of a box (SURVEY.md section 8e).

The reference would scan a chromosome as one string (`c_scan_motif` over a list with one sequence
per chromosome, cscore.c:336-389).  Two paths produce the same sites bit for bit:

* resident (default): the genome is encoded once into HBM (`genome.DeviceGenome`, 0.375 B/bp) and
  each chunk is a position RANGE of a resident chromosome (`msb_scan_ranges`): only windows that
  start inside the range are scored, and they read on into the rest of the chromosome, so no
  overlap is shipped and nothing is scored twice.  Chunks are dealt round-robin to the ranks.
* streamed (`resident=False`): a chunk is fetched from the host genome with a right overlap of
  (longest motif - 1) bases; the device drops sites whose start lies in the overlap
  (`msb_seqs_set_start_limit`).  Chunks are dealt to ranks longest-first (`shard.assign_lpt`).

Ranks never exchange data -- the only cross-rank step is the caller's gather of the per-motif
counts / site arrays.
"""
import ctypes
import time

import numpy as np

from . import _lib, engine, shard

_STRAND_ARG = {"+": 1, "-": 2, "both": 3}


class GenomeSites:
    """Sites of a genome-wide scan in the reference's order: motif, chromosome (sorted names, the
    order of `Genome.chroms`), start, forward before reverse."""

    def __init__(self, chroms, n_motifs, counts, motif, chrom_idx, start, score, strand):
        self.chroms = list(chroms)
        self.n_motifs = n_motifs
        self.counts = counts
        self._motif = motif          # None: built from the counts on first use (32 M entries for an hg19 share)
        self.chrom_idx, self.start, self.score, self.strand = chrom_idx, start, score, strand

    @property
    def motif(self):
        """Motif index of every site (the arrays are motif-major: `offsets` delimit the motifs)."""
        if self._motif is None:
            self._motif = np.repeat(np.arange(self.n_motifs, dtype=np.int32), self.counts if len(self.start) else 0)
        return self._motif

    @property
    def offsets(self):
        off = np.zeros(self.n_motifs + 1, dtype=np.int64)
        if len(self.start):
            np.cumsum(self.counts, out=off[1:])
        return off

    def __len__(self):
        return int(self.counts.sum())


def _merge_parts(parts, n_motifs):
    """Per-batch motif-major results -> one motif-major list.  Batches are scanned in ascending
    (chromosome, start) order and never overlap, so motif m's sites are the concatenation of its
    slice of every batch: no sort."""
    if not parts:
        return (np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float64),
                np.zeros(0, np.int8))
    if len(parts) == 1:
        c, cidx, start, score, strand = parts[0]
        return None, cidx, start, score, strand
    counts = np.stack([p[0] for p in parts])                  # [batch][motif]
    offs = np.zeros((len(parts), n_motifs + 1), dtype=np.int64)
    np.cumsum(counts, axis=1, out=offs[:, 1:])
    total = int(counts.sum())
    out_off = np.zeros(n_motifs + 1, dtype=np.int64)
    np.cumsum(counts.sum(axis=0), out=out_off[1:])
    cidx, start = np.empty(total, np.int32), np.empty(total, np.int32)
    score, strand = np.empty(total, np.float64), np.empty(total, np.int8)
    at = out_off[:-1].copy()
    for b, (_, c, s, sc, st) in enumerate(parts):
        for m in np.nonzero(counts[b])[0]:
            a, e = offs[b, m], offs[b, m + 1]
            d = at[m]
            cidx[d:d + e - a], start[d:d + e - a] = c[a:e], s[a:e]
            score[d:d + e - a], strand[d:d + e - a] = sc[a:e], st[a:e]
            at[m] += e - a
    return None, cidx, start, score, strand


def plan_ranges(chrom_sizes, chunk_bp, world=1, rank=0):
    """This rank's (chrom, start, end) ranges for the resident path: chromosomes in the given
    order cut every `chunk_bp` window starts, dealt round-robin (chunk k -> rank k % world).
    Ascending (chromosome, start) order within a rank."""
    out = []
    k = 0
    for chrom, size in chrom_sizes.items():
        for start in range(0, size, chunk_bp):
            if k % world == rank:
                out.append((chrom, start, min(start + chunk_bp, size)))
            k += 1
    return out


def scan_genome_resident(dgenome, pwms, p_value="1e-4", strand="both", chunk_bp=1 << 22, batch_bp=1 << 29,
                         world=1, rank=0, collect_sites=True, cutoffs=None, motifs=None, stats=None):
    """Range scan of a `genome.DeviceGenome`.  `motifs`: an engine.MotifSet to reuse (cutoffs set);
    `stats`: a dict that receives the summed device milliseconds per phase and the batch count."""
    ctx = dgenome.ctx
    matrices = [getattr(pwm, "matrix", pwm) for pwm in pwms]
    own_motifs = motifs is None
    if own_motifs:
        if cutoffs is None:
            cutoffs = [pwm.cutoffs[p_value] for pwm in pwms]
        motifs = engine.MotifSet(ctx, matrices, cutoffs)
    chroms = list(dgenome.chroms)
    sizes = {c: dgenome.chrom_sizes[c] for c in chroms}
    ranges = plan_ranges(sizes, chunk_bp, world, rank)
    counts = np.zeros(len(matrices), dtype=np.int64)
    parts, held = [], []
    try:
        i = 0
        while i < len(ranges):
            batch, total = [], 0
            while i < len(ranges) and (not batch or total + ranges[i][2] - ranges[i][1] <= batch_bp):
                c, a, e = ranges[i]
                if batch and batch[-1][0] == dgenome.chrom_index[c] and batch[-1][2] == a:
                    batch[-1][2] = e                      # adjacent chunks of one chromosome: one range
                else:
                    batch.append([dgenome.chrom_index[c], a, e])
                total += e - a
                i += 1
            if collect_sites:
                res = engine.scan_ranges(ctx, motifs, dgenome.seqs, _STRAND_ARG[strand], batch)
                counts += res.counts
                # the arrays stay views into the result's pinned block (kept alive by `held`): no host copy
                parts.append((res.counts.copy(), res.seq_idx, res.start, res.score, res.strand))
                held.append(res)
            else:
                engine.scan_ranges_device(ctx, motifs, dgenome.seqs, _STRAND_ARG[strand], batch)
                counts += ctx.site_counts(len(matrices))
            if stats is not None:
                t = ctx.timings()
                for k in ("prefilter", "exact", "order", "d2h"):
                    stats[k] = stats.get(k, 0.0) + t[k]
                stats["batches"] = stats.get("batches", 0) + 1
    finally:
        if own_motifs:
            motifs.close()
    motif, cidx, start, score, strnd = _merge_parts(parts, len(matrices))
    out = GenomeSites(chroms, len(matrices), counts, motif, cidx, start, score, strnd)
    if len(held) == 1:
        out._result = held[0]        # single batch: the site arrays ARE the pinned result block
    else:
        for res in held:
            res.close()
    return out


# ------------------------------------------------------------------------------------------------
# Sharded genome scan: several GPUs of one process (one host thread + one context per GPU) and / or
# several processes (world, rank), over a host `genome.PackedGenome`.
# ------------------------------------------------------------------------------------------------
class Unit:
    """A contiguous run of 32-base blocks [block0, block1) of the packed genome, uploaded with `halo`
    extra blocks behind it, as the sequences `pieces` = (chromosome index, start, owned end, fetched end):
    windows that START in [start, owned end) belong to the unit and may read on to `fetched end`."""
    __slots__ = ("block0", "block1", "upload1", "pieces")

    def __init__(self, block0, block1, upload1, pieces):
        self.block0, self.block1, self.upload1, self.pieces = block0, block1, upload1, pieces

    @property
    def owned_bp(self):
        return sum(b - a for _, a, b, _ in self.pieces)


def plan_units(block_off, chrom_sizes, n_shares, unit_blocks, halo_bases, work_prefix=None, taper=False):
    """Cut the packed block space [0, B) into `n_shares` contiguous shares of (almost) equal size and every
    share into units of at most `unit_blocks` blocks.  Returns a list (per share) of lists of `Unit`.
    Every base of every chromosome is owned by exactly one unit; share and unit boundaries are multiples
    of 32 bases inside a chromosome, so a unit's planes are a plain slice of the genome's.

    `work_prefix` (B + 1 cumulative per-block weights, e.g. `PackedGenome.work_prefix()`): shares are cut at
    equal WORK instead of equal size -- position tiles that hold nothing but N cost the device nothing, and
    assembly gaps are not spread evenly over a genome."""
    n_blocks = int(block_off[-1])
    halo = (max(int(halo_bases), 0) + 31) // 32
    if work_prefix is not None and n_blocks:
        total = float(work_prefix[-1])
        cuts = [int(np.searchsorted(work_prefix, total * k / n_shares, side="left")) for k in range(n_shares + 1)]
        cuts[0], cuts[-1] = 0, n_blocks
        cuts = [min(max(c, 0), n_blocks) for c in cuts]
        for k in range(1, len(cuts)):
            cuts[k] = max(cuts[k], cuts[k - 1])
    else:
        cuts = [n_blocks * k // n_shares for k in range(n_shares + 1)]
    shares = []
    for k in range(n_shares):
        s0, s1 = cuts[k], cuts[k + 1]
        n_units = max(1, -(-(s1 - s0) // max(int(unit_blocks), 1)))
        bounds = [s0 + (s1 - s0) * u // n_units for u in range(n_units + 1)]
        if taper and bounds[-1] - bounds[-2] >= 4096:
            # the copy-back of a share's LAST unit is the one transfer no scan hides: cut that unit into 1/2, 1/4, 1/4
            a, b = bounds[-2], bounds[-1]
            bounds[-1:] = [a + (b - a) // 2, a + 3 * (b - a) // 4, b]
        units = []
        for u0, u1 in zip(bounds[:-1], bounds[1:]):
            if u1 <= u0:
                continue
            pieces = []
            c = int(np.searchsorted(block_off, u0, side="right")) - 1
            upload1 = u1
            while c < len(chrom_sizes) and block_off[c] < u1:
                cb0, size = int(block_off[c]), int(chrom_sizes[c])
                a = (max(u0, cb0) - cb0) * 32
                b = min((min(u1, int(block_off[c + 1])) - cb0) * 32, size)
                f = min(b + halo * 32, size)
                if b > a:
                    pieces.append((c, a, b, f))
                    upload1 = max(upload1, cb0 + (f + 31) // 32)
                c += 1
            units.append(Unit(u0, u1, upload1, pieces))
        shares.append(units)
    return shares


class ShardedSites(GenomeSites):
    """GenomeSites over the per-unit results of a sharded scan: the per-motif counts are there at once,
    the site arrays are gathered on first use (`msb_merge_motif_major`: per motif, unit after unit in
    genome order -- a copy, no sort) and unit-local (piece, offset) coordinates become (chromosome, start)."""

    def __init__(self, chroms, n_motifs, counts, parts):
        # parts: list of (ScanResult, piece chromosome index array, piece start array), in genome order
        self.chroms = list(chroms)
        self.n_motifs = n_motifs
        self.counts = counts
        self._motif = None
        self._parts = parts          # chrom_idx / start / score / strand appear on first use (__getattr__)
        self._merged = False

    def _merge(self):
        if self._merged:
            return
        parts = [p for p in self._parts if p[0].n_sites]
        if not parts:
            self.chrom_idx, self.start = np.zeros(0, np.int32), np.zeros(0, np.int32)
            self.score, self.strand = np.zeros(0, np.float64), np.zeros(0, np.int8)
        else:
            cnt = np.stack([p[0].counts for p in parts])
            if all(p[0].compact() is not None for p in parts):      # 12-byte sites: decoded while they are gathered
                self.chrom_idx, self.start, self.score, self.strand = engine.merge_sites_compact(
                    cnt, [p[0] for p in parts], seq_to_group=[p[1] for p in parts], seq_offset=[p[2] for p in parts])
            else:
                self.chrom_idx, self.start, self.score, self.strand = engine.merge_sites(
                    cnt, [p[0].seq_idx for p in parts], [p[0].start for p in parts], [p[0].score for p in parts],
                    [p[0].strand for p in parts], seq_to_group=[p[1] for p in parts], seq_offset=[p[2] for p in parts])
        fix = self.__dict__.get("_fix")
        if fix is not None:
            dev_counts = np.sum([p[0].counts for p in self._parts], axis=0)
            self._apply_fix(fix, dev_counts)
        for p in self._parts:
            p[0].close()
        self._parts = []
        self._merged = True

    def _apply_fix(self, fix, dev_counts):
        """Sites that boundary stitching removed or restored (GenomeScanner with remove_dup): the arrays hold the
        per-piece de-duplicated sites; entries are deleted and inserted at their (motif, chromosome, start, strand)
        place."""
        off = np.zeros(len(dev_counts) + 1, dtype=np.int64)
        np.cumsum(dev_counts, out=off[1:])

        def key(chrom, start, strand):
            return (chrom.astype(np.int64) << 34) | (start.astype(np.int64) << 2) | strand.astype(np.int64)
        pos = np.zeros(len(fix["motif"]), dtype=np.int64)
        fkey = key(fix["chrom"], fix["start"], fix["strand"])
        for m in np.unique(fix["motif"]):
            a, b = off[m], off[m + 1]
            sel = fix["motif"] == m
            pos[sel] = a + np.searchsorted(key(self.chrom_idx[a:b], self.start[a:b], self.strand[a:b]), fkey[sel])
        rm = np.sort(pos[~fix["add"]])
        add = np.flatnonzero(fix["add"])
        add = add[np.lexsort((fkey[add], fix["motif"][add]))]
        at = pos[add] - np.searchsorted(rm, pos[add], side="left")
        for name, val in (("chrom_idx", fix["chrom"]), ("start", fix["start"]), ("score", fix["score"]), ("strand", fix["strand"])):
            arr = np.delete(getattr(self, name), rm)
            setattr(self, name, np.insert(arr, at, val[add].astype(arr.dtype)))

    def __getattr__(self, name):
        if name in ("chrom_idx", "start", "score", "strand") and not self.__dict__.get("_merged", True):
            self._merge()
            return self.__dict__[name]
        raise AttributeError(name)

    def close(self):
        for p in self._parts:
            p[0].close()
        self._parts = []


def _greedy_keep(start, score, length):
    """Keep flags of the reference's greedy de-duplication (scanner.py:156-168) over one chain of one strand."""
    keep = np.zeros(len(start), dtype=bool)
    cur = -1
    for i in range(len(start)):
        if cur >= 0 and start[i] - start[cur] < length:
            if score[cur] >= score[i]:
                continue
            keep[cur] = False
        keep[i] = True
        cur = i
    return keep


def stitch_boundaries(rec, piece_chrom, lengths):
    """Chains of overlapping sites cut by piece boundaries, resolved as if the chromosome had been one sequence.

    `rec`: the boundary sites of every piece (`Context.boundary_sites`), with `piece` (global piece index, pieces
    in genome order) and `gstart` (start on the chromosome) added; `piece_chrom[p]`: chromosome of piece p, and
    consecutive pieces of one chromosome are adjacent.  The tail chain of a piece is joined with the head chain of
    the next piece when they are less than a motif length apart; a chain that is both the head and the tail of its
    piece is carried on to the next boundary.  Every joined chain gets the greedy rule again.  Returns the indices
    into `rec` whose keep flag changes, and the number of chains that crossed a boundary."""
    changed, n_joined = [], 0
    if not len(rec["motif"]):
        return np.zeros(0, dtype=np.int64), 0
    order = np.lexsort((rec["gstart"], rec["piece"], rec["strand"], rec["motif"]))
    motif, strand, piece = rec["motif"][order], rec["strand"][order], rec["piece"][order]
    gstart, score, flags = rec["gstart"][order], rec["score"][order], rec["flags"][order]
    bounds = np.flatnonzero(np.diff(motif) | np.diff(strand) | np.diff(piece)) + 1
    groups = np.split(np.arange(len(order)), bounds)       # one (motif, strand, piece) each, in genome order

    def resolve(chain):
        nonlocal n_joined
        if len(chain) < 2 or piece[chain[0]] == piece[chain[-1]]:
            return                                        # one piece: the device's flags are final
        n_joined += 1
        idx = np.asarray(chain)
        keep = _greedy_keep(gstart[idx], score[idx], lengths[motif[idx[0]]])
        changed.extend(order[idx[keep != ((flags[idx] & 1) == 1)]].tolist())

    carry, key = [], None
    for g in groups:
        first = g[0]
        head = [i for i in g if flags[i] & 2]
        tail = [i for i in g if flags[i] & 4]
        whole = bool(head) and bool(flags[head[0]] & 4)    # one chain from the piece's start to its end
        this = (motif[first], strand[first], piece_chrom[piece[first]])
        if carry and key == this and head and gstart[head[0]] - gstart[carry[-1]] < lengths[motif[first]]:
            if whole:
                carry = carry + head
                continue
            resolve(carry + head)
        else:
            resolve(carry)
        carry, key = tail, this
    resolve(carry)
    return np.asarray(changed, dtype=np.int64), n_joined


class GenomeScanner:
    """Genome-wide scan of a host `PackedGenome` on several GPUs: `devices` of THIS process (one host thread
    and one context per device; the C calls drop the GIL) times `world` processes (`rank` = this one).  The
    packed genome is cut into world x len(devices) contiguous shares; a share is processed in units that
    are uploaded (0.375 B/bp, asynchronously, on the copy stream), scanned, and whose sites are copied back
    (asynchronously, on the d2h stream) while the next unit is being scanned.  No device ever talks to
    another one: the only gather is the host-side sum of the per-motif counts and the per-motif
    concatenation of the site arrays (SURVEY.md section 8e; the reference's analogue is its in-process
    thread pool over motifs, cscore.c:323-328, 425-436)."""

    def __init__(self, pg, pwms, cutoffs=None, p_value="1e-4", strand="both", devices=None, world=1, rank=0,
                 unit_bp=1 << 26, resident=False, contexts=None, compact=True, remove_dup=False):
        if remove_dup and int(world) > 1:
            raise ValueError("GenomeScanner: remove_dup=True needs the whole genome in one process (world = 1)")
        self.pg = pg
        # the reference's adjacent-site de-duplication over whole chromosomes: per piece on the device, the chains
        # that cross a unit or share boundary stitched on the host (stitch_boundaries)
        self.remove_dup = bool(remove_dup)
        self.matrices = [getattr(pwm, "matrix", pwm) for pwm in pwms]
        if cutoffs is None:
            cutoffs = [pwm.cutoffs[p_value] for pwm in pwms]
        self.cutoffs = np.ascontiguousarray(np.asarray(cutoffs, dtype=np.float64))
        self.strand = _STRAND_ARG[strand]
        if contexts is not None:                  # the caller's contexts (e.g. on its own streams), one per device
            devices = [c.device for c in contexts]
        self.devices = list(devices) if devices is not None else [0]
        self.world, self.rank = int(world), int(rank)
        lmax = max([np.asarray(m).shape[1] for m in self.matrices] + [1])
        sizes = [pg.chrom_sizes[c] for c in pg.chroms]
        n_shares = self.world * len(self.devices)
        work = pg.work_prefix() if n_shares > 1 and hasattr(pg, "work_prefix") else None
        shares = plan_units(pg.block_off, sizes, n_shares, max(int(unit_bp) // 32, 1), lmax - 1, work_prefix=work, taper=True)
        self.shares = shares[self.rank * len(self.devices):(self.rank + 1) * len(self.devices)]
        self.ctxs = list(contexts) if contexts is not None else [engine.default_context(d) for d in self.devices]
        self.motifs = [engine.MotifSet(ctx, self.matrices, self.cutoffs) for ctx in self.ctxs]
        self.resident = [None] * len(self.devices)     # per device: the uploaded units, kept between scans
        self.keep_resident = bool(resident)
        self.compact = bool(compact)          # 12-byte site records over PCIe (MSB_SCAN_COMPACT)
        self.last_stats = None

    def _upload(self, ctx, unit, async_):
        codes, nmask = self.pg.planes(unit.block0, unit.upload1)
        return engine.SequenceSet.from_packed(ctx, [f - a for _, a, _, f in unit.pieces], codes, nmask, async_=async_)

    def _scan_share(self, k, collect_sites, order_sites=False):
        ctx, motifs, units = self.ctxs[k], self.motifs[k], self.shares[k]
        if len(self.devices) > 1:
            _lib.bind_thread_near(ctx.device)     # worker thread of one GPU: stay on that GPU's side of the host
        n_motifs = len(self.matrices)
        counts = np.zeros(n_motifs, dtype=np.int64)
        parts, stats, cells, bnd = [], {}, [], []
        kept = self.resident[k]
        nxt = None
        try:
            for i, unit in enumerate(units):
                if kept is not None:
                    sset = kept[i]
                else:
                    sset = nxt if nxt is not None else self._upload(ctx, unit, True)
                    nxt = None
                    if i + 1 < len(units):        # the next unit's planes travel while this one is scanned
                        nxt = self._upload(ctx, units[i + 1], True)
                ranges = [(j, 0, b - a) for j, (_, a, b, _) in enumerate(unit.pieces)]
                with ctx._lock:   # the counts / timings read below belong to THIS scan even if the context is shared
                    if collect_sites:
                        res = engine.scan_ranges(ctx, motifs, sset, self.strand, ranges, async_=True, compact=self.compact,
                                                 remove_dup=self.remove_dup)
                        parts.append((res, np.array([p[0] for p in unit.pieces]), np.array([p[1] for p in unit.pieces])))
                    else:
                        engine.scan_ranges_device(ctx, motifs, sset, self.strand, ranges, counts_only=not order_sites,
                                                  remove_dup=self.remove_dup)
                        counts += ctx.site_counts(n_motifs)
                    t = ctx.timings()
                    c = ctx.counters()
                    if self.remove_dup:
                        t0 = time.perf_counter()
                        cells.append(ctx.cell_stats(n_motifs, len(unit.pieces)))
                        bnd.append(ctx.boundary_sites())
                        stats["boundary_read_s"] = stats.get("boundary_read_s", 0.0) + time.perf_counter() - t0
                for name in ("prefilter", "exact", "order"):
                    stats[name] = stats.get(name, 0.0) + t[name]
                for name in ("launches", "prefilter_launches", "candidates", "hits"):
                    stats[name] = stats.get(name, 0) + c[name]
                if self.keep_resident and kept is None:
                    self.resident[k] = (self.resident[k] or []) + [sset]
                elif kept is None:
                    sset.close()
            for res, _, _ in parts:
                counts += res.counts            # waits for that unit's copy
        finally:
            if nxt is not None:
                nxt.close()
        stats["units"] = len(units)
        return counts, parts, stats, cells, bnd

    def scan(self, collect_sites=True, order_sites=False):
        """One pass over this process's shares.  Returns a `ShardedSites` (`collect_sites=False`: per-motif
        counts only -- MSB_SCAN_COUNTS, nothing but 8 bytes per motif and unit leaves a device;
        `order_sites=True` then still orders the sites on the device, as a measurement of that stage).

        With `remove_dup` the sites are the reference's de-duplicated ones over whole chromosomes, and the result
        also carries `cell_counts` / `cell_best` (int64 / float64 [n_motifs, n_chroms], NaN where a cell is empty):
        the sites and best score of every (motif, chromosome), which is all the two result tables need.  Without
        `collect_sites` no site array leaves a device."""
        n = len(self.devices)
        if n == 1:
            outs = [self._scan_share(0, collect_sites, order_sites)]
        else:
            import concurrent.futures
            with concurrent.futures.ThreadPoolExecutor(max_workers=n) as pool:
                outs = list(pool.map(lambda k: self._scan_share(k, collect_sites, order_sites), range(n)))
        counts = np.sum([o[0] for o in outs], axis=0)
        parts = [p for o in outs for p in o[1]]
        self.last_stats = [o[2] for o in outs]
        if not self.remove_dup:
            return ShardedSites(self.pg.chroms, len(self.matrices), counts, parts)
        units = [u for share in self.shares for u in share]
        return self._stitched(units, [c for o in outs for c in o[3]], [b for o in outs for b in o[4]], parts)

    def _stitched(self, units, cells, bnd, parts):
        """Per-piece de-duplicated results of every unit (genome order) -> whole-chromosome results."""
        t0 = time.perf_counter()
        n_motifs, n_chroms = len(self.matrices), len(self.pg.chroms)
        lengths = np.array([np.asarray(m).shape[1] for m in self.matrices], dtype=np.int64)
        piece_chrom = np.array([p[0] for u in units for p in u.pieces], dtype=np.int64)
        piece_a = np.array([p[1] for u in units for p in u.pieces], dtype=np.int64)
        first = np.cumsum([0] + [len(u.pieces) for u in units])
        rec = {name: np.concatenate([b[name] for b in bnd]) if bnd else np.zeros(0)
               for name in ("motif", "seq_idx", "start", "score", "strand", "flags")}
        rec["piece"] = np.concatenate([b["seq_idx"].astype(np.int64) + first[i] for i, b in enumerate(bnd)]) if bnd else np.zeros(0, np.int64)
        rec["gstart"] = piece_a[rec["piece"]] + rec["start"] if len(rec["piece"]) else np.zeros(0, np.int64)
        changed, n_joined = stitch_boundaries(rec, piece_chrom, lengths)
        # per (motif, piece) -> per (motif, chromosome)
        cell_counts = np.zeros((n_motifs, n_chroms), dtype=np.int64)
        cell_best = np.full((n_motifs, n_chroms), np.nan)
        for (cnt, best), u in zip(cells, units):
            for j, p in enumerate(u.pieces):
                cell_counts[:, p[0]] += cnt[:, j]
                hit = cnt[:, j] > 0
                cell_best[hit, p[0]] = np.fmax(cell_best[hit, p[0]], best[hit, j])
        add = np.where((rec["flags"][changed] & 1) == 0, 1, -1) if len(changed) else np.zeros(0, np.int64)
        np.add.at(cell_counts, (rec["motif"][changed], piece_chrom[rec["piece"][changed]]), add)
        counts = cell_counts.sum(axis=1)
        out = ShardedSites(self.pg.chroms, n_motifs, counts, parts)
        out.cell_counts, out.cell_best = cell_counts, cell_best
        if len(changed) and parts:
            out._fix = dict(motif=rec["motif"][changed], chrom=piece_chrom[rec["piece"][changed]].astype(np.int32),
                            start=rec["gstart"][changed].astype(np.int32), score=rec["score"][changed],
                            strand=rec["strand"][changed], add=add > 0)
        self.last_stitch = {"boundary_sites": int(len(rec["motif"])), "joined_chains": n_joined,
                            "corrections": int(len(changed)), "removed": int((add < 0).sum()), "stitch_s": time.perf_counter() - t0}
        return out

    def close(self):
        for kept in self.resident:
            for sset in kept or []:
                sset.close()
        self.resident = [None] * len(self.devices)
        for m in self.motifs:
            m.close()
        self.motifs = []


def plan_chunks(chrom_sizes, chunk_bp, halo, world=1, rank=0):
    """This rank's chunks as (chrom, start, end, fetch_end), in (chromosome, start) order."""
    chunks = shard.genome_chunks(chrom_sizes, chunk_bp, halo)
    if world > 1:
        owner, _ = shard.assign_lpt([c[2] - c[1] for c in chunks], world)
        chunks = [c for c, o in zip(chunks, owner) if o == rank]
    return chunks


def scan_genome(genome, pwms, p_value="1e-4", strand="both", chunk_bp=1 << 22, batch_bp=1 << 28,
                ctx=None, world=1, rank=0, collect_sites=True, cutoffs=None, resident=True, devices=None, remove_dup=False):
    """Scan all chromosomes of `genome` (anything with `.chroms`, `.chrom_sizes`, `.fetch_bytes`).

    `devices=[...]`: use these GPUs of this process together (`GenomeScanner`; the genome is packed on
    the host first unless it already is a `genome.PackedGenome`); sites come back gathered in the
    reference's order, identical to the one-GPU result.

    Returns a GenomeSites for this rank's chunks (`collect_sites=False`: counts only, the site
    arrays stay empty and nothing but the counts leaves the device).  A `genome.DeviceGenome` is
    scanned in place; a host genome is first made resident (`resident=True`, the default) or
    streamed chunk by chunk with overlaps (`resident=False`).

    `remove_dup=True`: the reference's de-duplication over whole chromosomes, always through `GenomeScanner`
    (a host genome is packed first); a `genome.DeviceGenome` or `resident=False` is an error."""
    from .genome import PackedGenome
    if remove_dup:
        if hasattr(genome, "chrom_index") and hasattr(genome, "seqs"):
            raise ValueError("scan_genome: remove_dup=True scans a host or packed genome (GenomeScanner), not a DeviceGenome")
        if not resident:
            raise ValueError("scan_genome: remove_dup=True is not available on the streamed path (resident=False)")
    if devices is not None or isinstance(genome, PackedGenome) or remove_dup:
        devices = list(devices) if devices is not None else [ctx.device if ctx is not None else 0]
        pg = genome if isinstance(genome, PackedGenome) else PackedGenome.from_genome(genome, engine.default_context(devices[0]))
        gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, p_value=p_value, strand=strand, devices=devices, world=world, rank=rank,
                           remove_dup=remove_dup)
        try:
            return gs.scan(collect_sites=collect_sites)
        finally:
            gs.close()
    if hasattr(genome, "chrom_index") and hasattr(genome, "seqs"):
        return scan_genome_resident(genome, pwms, p_value, strand, chunk_bp, batch_bp, world, rank,
                                    collect_sites, cutoffs)
    if resident:
        from .genome import DeviceGenome
        dg = DeviceGenome(genome, ctx or engine.default_context(0))
        try:
            return scan_genome_resident(dg, pwms, p_value, strand, chunk_bp, batch_bp, world, rank,
                                        collect_sites, cutoffs)
        finally:
            dg.close()
    if cutoffs is None:
        cutoffs = [pwm.cutoffs[p_value] for pwm in pwms]
    matrices = [getattr(pwm, "matrix", pwm) for pwm in pwms]
    lmax = max(np.asarray(m).shape[1] for m in matrices)
    ctx = ctx or engine.default_context(0)
    chroms = list(genome.chroms)
    chrom_id = {c: i for i, c in enumerate(chroms)}
    sizes = {c: genome.chrom_sizes[c] for c in chroms}
    chunks = plan_chunks(sizes, chunk_bp, lmax - 1, world, rank)
    motifs = engine.MotifSet(ctx, matrices, cutoffs)
    counts = np.zeros(len(matrices), dtype=np.int64)
    parts = []
    # one pinned staging buffer for the ASCII of a batch: chunks are copied into it once and go to
    # the device at full PCIe speed
    cap = max([f - a for _, a, _, f in chunks] + [1])
    cap = max(cap, min(batch_bp, sum(f - a for _, a, _, f in chunks)))
    pinned = ctypes.c_void_p()
    _lib.check(ctx._lib.msb_pinned_alloc(int(cap), ctypes.byref(pinned)))
    stage = np.ctypeslib.as_array(ctypes.cast(pinned, ctypes.POINTER(ctypes.c_uint8)), shape=(cap,))
    try:
        i = 0
        while i < len(chunks):
            batch, total = [], 0
            while i < len(chunks) and (not batch or total + chunks[i][3] - chunks[i][1] <= batch_bp):
                batch.append(chunks[i])
                total += chunks[i][3] - chunks[i][1]
                i += 1
            off = np.zeros(len(batch) + 1, dtype=np.int64)
            for k, (c, a, _, f) in enumerate(batch):
                piece = np.frombuffer(genome.fetch_bytes(c, a, f), dtype=np.uint8)
                off[k + 1] = off[k] + piece.size
                stage[off[k]:off[k + 1]] = piece
            sset = engine.SequenceSet(ctx, blob=stage[:off[-1]], seq_off=off)
            try:
                sset.set_start_limit([e - a for _, a, e, _ in batch])
                if collect_sites:
                    res = engine.scan(ctx, motifs, sset, _STRAND_ARG[strand])
                    counts += res.counts
                    cid = np.array([chrom_id[c] for c, _, _, _ in batch], dtype=np.int32)
                    base = np.array([a for _, a, _, _ in batch], dtype=np.int64)
                    parts.append((np.repeat(np.arange(len(matrices), dtype=np.int32), res.counts),
                                  cid[res.seq_idx], base[res.seq_idx] + res.start, res.score.copy(), res.strand.copy()))
                    res.close()
                else:
                    engine.scan_device(ctx, motifs, sset, _STRAND_ARG[strand])
                    counts += ctx.site_counts(len(matrices))
            finally:
                sset.close()
    finally:
        motifs.close()
        ctx._lib.msb_pinned_free(pinned)
    if parts:
        motif, cidx, start, score, strnd = (np.concatenate(x) for x in zip(*parts))
        order = np.lexsort((strnd, start, cidx, motif))
        motif, cidx, start, score, strnd = motif[order], cidx[order], start[order], score[order], strnd[order]
    else:
        motif, cidx = np.zeros(0, np.int32), np.zeros(0, np.int32)
        start, score, strnd = np.zeros(0, np.int64), np.zeros(0, np.float64), np.zeros(0, np.int8)
    return GenomeSites(chroms, len(matrices), counts, motif, cidx, start, score, strnd)
