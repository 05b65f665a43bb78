"""Handle classes over the C ABI (include/msb200.h): Context, MotifSet, SequenceSet, ScanResult.

These are the array-native entry points the host code (Scanner, cutoff builder, bench) uses; the
list-of-lists mirrors of the reference's extension methods live in motifscan_b200/motif/cscore.py.
"""
import ctypes
import threading

import numpy as np

from . import _lib
from ._lib import check, ptr

_default = {}
_default_lock = threading.Lock()


class Context:
    """One device, one stream, reusable scratch (msb_ctx)."""

    def __init__(self, device=0, stream=None):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        check(self._lib.msb_ctx_create(int(device), ctypes.c_void_p(stream or 0), ctypes.byref(self._h)))
        self.device = int(device)
        # an msb_ctx owns one stream and one set of scratch buffers: calls on it are serialised here so
        # that host threads sharing a context (e.g. two Scanners on default_context) cannot interleave
        self._lock = threading.RLock()

    def close(self):
        if self._h:
            self._lib.msb_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(self._lib.msb_ctx_sync(self._h))

    def set_option(self, name, value):
        """Tuning / test knob of this context only (msb_ctx_set_option; names in include/msb200.h)."""
        with self._lock:
            check(self._lib.msb_ctx_set_option(self._h, name.encode(), int(value)))

    def timings(self):
        """Device milliseconds per phase of the last call (CUDA events on the context's stream)."""
        a = np.zeros(len(_lib.T_NAMES), dtype=np.float64)
        check(self._lib.msb_ctx_timings(self._h, ptr(a, ctypes.c_double), len(a)))
        return dict(zip(_lib.T_NAMES, a.tolist()))

    def site_counts(self, n_motifs):
        """Per-motif site counts of the last `scan_device` on this context."""
        out = np.zeros(max(n_motifs, 1), dtype=np.int64)
        with self._lock:
            check(self._lib.msb_scan_device_counts(self._h, ptr(out, ctypes.c_int64), int(n_motifs)))
        return out[:n_motifs]

    def region_counts(self, n_motifs):
        """Per motif, the number of sequences with at least one site in the last `scan_device` on this
        context (what stats.motif_enrichment counts), reduced on the device."""
        out = np.zeros(max(n_motifs, 1), dtype=np.int64)
        with self._lock:
            check(self._lib.msb_scan_device_region_counts(self._h, ptr(out, ctypes.c_int64), int(n_motifs)))
        return out[:n_motifs]

    def boundary_sites(self):
        """Boundary chains of the last de-duplicated range scan on this context (msb_scan_device_boundary_sites):
        a dict of equal-length arrays motif, seq_idx, start, score, strand, flags (bit 0 kept, bit 1 head chain,
        bit 2 tail chain)."""
        n = ctypes.c_int64(0)
        with self._lock:
            check(self._lib.msb_scan_device_boundary_sites(self._h, 0, ctypes.byref(n), None, None, None, None, None, None))
            k = n.value
            out = dict(motif=np.zeros(k, np.int32), seq_idx=np.zeros(k, np.int32), start=np.zeros(k, np.int32),
                       score=np.zeros(k, np.float64), strand=np.zeros(k, np.int8), flags=np.zeros(k, np.int8))
            if k:
                check(self._lib.msb_scan_device_boundary_sites(
                    self._h, k, ctypes.byref(n), ptr(out["motif"], ctypes.c_int32), ptr(out["seq_idx"], ctypes.c_int32),
                    ptr(out["start"], ctypes.c_int32), ptr(out["score"], ctypes.c_double), ptr(out["strand"], ctypes.c_int8),
                    ptr(out["flags"], ctypes.c_int8)))
        return out

    def cell_stats(self, n_motifs, n_seqs):
        """(counts int64[n_motifs, n_seqs], best float64[n_motifs, n_seqs], NaN where empty) of the last scan on this
        context, reduced on the device (msb_scan_device_cell_stats)."""
        counts = np.zeros((n_motifs, n_seqs), dtype=np.int64)
        best = np.full((n_motifs, n_seqs), np.nan)
        if counts.size:
            with self._lock:
                check(self._lib.msb_scan_device_cell_stats(self._h, int(n_motifs), int(n_seqs), ptr(counts, ctypes.c_int64),
                                                           ptr(best, ctypes.c_double)))
        return counts, best

    def pair_counts(self, n_motifs, n_seqs):
        """int64[n_motifs, n_motifs]: the number of sequences with a final site of both motifs in the last scan on this
        context (the diagonal: with a site of the motif), from the (motif, sequence) bit matrix on the device
        (msb_scan_device_pair_counts)."""
        out = np.zeros((max(n_motifs, 1), max(n_motifs, 1)), dtype=np.int64)
        with self._lock:
            check(self._lib.msb_scan_device_pair_counts(self._h, int(n_motifs), int(n_seqs), ptr(out, ctypes.c_int64)))
        return out[:n_motifs, :n_motifs]

    def spacing(self, motifs, anchors, max_offset):
        """int64[n_anchors, n_motifs, 2, 2 max_offset + 1]: partner sites around each anchor motif's sites in the last
        scan on this context, by partner motif, orientation (0 same strand, 1 opposite) and offset -max_offset ..
        max_offset in the anchor's frame (msb_scan_device_spacing)."""
        a = np.ascontiguousarray(np.asarray(anchors, dtype=np.int32).reshape(-1))
        d = int(max_offset)
        ok = 1 <= len(a) <= 16 and 0 <= d <= 500
        out = np.zeros((len(a), motifs.n, 2, 2 * d + 1) if ok else 1, dtype=np.int64)
        with self._lock:
            check(self._lib.msb_scan_device_spacing(self._h, motifs._h, len(a), ptr(a if len(a) else np.zeros(1, np.int32),
                                                                                     ctypes.c_int32), d, ptr(out, ctypes.c_int64)))
        return out

    def centrality(self, motifs, mid2, bin, half_bins):
        """(hist_all, hist_best), int64[n_motifs, 2 half_bins + 1] each: the last scan's final sites on this context by
        bin floor((d2 + bin) / (2 bin)), d2 = 2 start + L - mid2[s], for bins -half_bins..half_bins; hist_best counts
        the best site of each (motif, sequence) cell.  mid2[s] < 0 leaves sequence s out; len(mid2) must be the
        scanned set's sequence count (msb_scan_device_centrality)."""
        m = np.ascontiguousarray(np.asarray(mid2, dtype=np.int32).reshape(-1))
        h = int(half_bins)
        ok = h >= 0 and motifs.n * (2 * h + 1) <= _lib.CENTRALITY_MAX_CELLS
        hist_all = np.zeros((motifs.n, 2 * h + 1) if ok else 1, dtype=np.int64)
        hist_best = np.zeros_like(hist_all)
        with self._lock:
            check(self._lib.msb_scan_device_centrality(self._h, motifs._h, len(m), ptr(m if len(m) else np.zeros(1, np.int32),
                                                                                        ctypes.c_int32), int(bin), h,
                                                       ptr(hist_all, ctypes.c_int64), ptr(hist_best, ctypes.c_int64)))
        return hist_all, hist_best

    def counters(self):
        a = np.zeros(len(_lib.C_NAMES), dtype=np.int64)
        check(self._lib.msb_ctx_counters(self._h, ptr(a, ctypes.c_int64), len(a)))
        return dict(zip(_lib.C_NAMES, a.tolist()))


def default_context(device=0):
    with _default_lock:
        if device not in _default:
            _default[device] = Context(device)
        return _default[device]


class MotifSet:
    """Device-resident PWMs + cutoffs (msb_motifs)."""

    def __init__(self, ctx, pwms, cutoffs=None):
        self.ctx = ctx
        self._lib = ctx._lib
        lens, mats, mat_off = _lib.flatten_pwms(pwms)
        self.lengths = lens
        self.n = len(lens)
        cut = None
        if cutoffs is not None:
            cut = np.ascontiguousarray(np.asarray(cutoffs, dtype=np.float64))
            if cut.shape != (self.n,):
                raise ValueError("cutoffs must have one entry per PWM")
        self._h = ctypes.c_void_p()
        check(self._lib.msb_motifs_create(ctx._h, self.n, ptr(lens, ctypes.c_int32), ptr(mats, ctypes.c_double),
                                          ptr(mat_off, ctypes.c_int64),
                                          ptr(cut, ctypes.c_double) if cut is not None else None,
                                          ctypes.byref(self._h)))

    def set_cutoffs(self, cutoffs):
        cut = np.ascontiguousarray(np.asarray(cutoffs, dtype=np.float64))
        if cut.shape != (self.n,):
            raise ValueError("cutoffs must have one entry per PWM")
        check(self._lib.msb_motifs_set_cutoffs(self._h, ptr(cut, ctypes.c_double)))

    def max_raw(self):
        out = np.zeros(max(self.n, 1), dtype=np.float64)
        check(self._lib.msb_motifs_max_raw(self._h, ptr(out, ctypes.c_double)))
        return out[:self.n]

    def close(self):
        if self._h:
            self._lib.msb_motifs_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SequenceSet:
    """Device-resident packed sequences (msb_seqs): 2-bit codes + N mask."""

    def __init__(self, ctx, seqs=None, blob=None, seq_off=None, _handle=None):
        self.ctx = ctx
        self._lib = ctx._lib
        if _handle is not None:
            self._h = _handle
            n, bp = ctypes.c_int64(0), ctypes.c_int64(0)
            check(self._lib.msb_seqs_count(self._h, ctypes.byref(n), ctypes.byref(bp)))
            self.n, self.total_bp = n.value, bp.value
            lens = np.zeros(max(self.n, 1), dtype=np.int64)
            check(self._lib.msb_seqs_lengths(self._h, ptr(lens, ctypes.c_int64)))
            self.seq_off = np.zeros(self.n + 1, dtype=np.int64)
            np.cumsum(lens[:self.n], out=self.seq_off[1:])
            return
        if seqs is not None:
            blob, seq_off = _lib.flatten_seqs(seqs)
        blob = np.ascontiguousarray(blob, dtype=np.uint8) if not isinstance(blob, np.ndarray) else blob
        seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
        self.n = len(seq_off) - 1
        self.total_bp = int(seq_off[-1])
        self.seq_off = seq_off
        self._h = ctypes.c_void_p()
        data = blob.ctypes.data if blob.size else None
        with self.ctx._lock:
            check(self._lib.msb_seqs_from_ascii(ctx._h, self.n, ctypes.c_void_p(data), ptr(seq_off, ctypes.c_int64),
                                                ctypes.byref(self._h)))

    @classmethod
    def from_packed(cls, ctx, lens, codes, nmask, async_=False):
        """Sequences that are already packed in the library's layout (msb_seqs_from_packed): `codes`
        uint32[2 B], `nmask` uint32[B] with B = sum ceil(len / 32); 0.375 B/bp cross PCIe and nothing is
        encoded.  The arrays may be views into a larger (pinned) buffer, e.g. a `genome.PackedGenome`.
        `async_`: the copy runs on the context's copy stream and overlaps a scan in progress."""
        lens = np.ascontiguousarray(np.asarray(lens, dtype=np.int64))
        n_blocks = int(((lens + 31) // 32).sum())
        codes = np.ascontiguousarray(codes, dtype=np.uint32)
        nmask = np.ascontiguousarray(nmask, dtype=np.uint32)
        if codes.size < 2 * n_blocks or nmask.size < n_blocks:
            raise ValueError("packed planes are shorter than the sequence lengths require")
        h = ctypes.c_void_p()
        with ctx._lock:
            check(ctx._lib.msb_seqs_from_packed(ctx._h, len(lens), ptr(lens, ctypes.c_int64),
                                                ctypes.c_void_p(codes.ctypes.data if n_blocks else 0),
                                                ctypes.c_void_p(nmask.ctypes.data if n_blocks else 0),
                                                _lib.MSB_SEQS_ASYNC if async_ else 0, ctypes.byref(h)))
        out = cls(ctx, _handle=h)
        out._planes = (codes, nmask) if async_ else None   # an asynchronous upload still reads them
        return out

    def to_packed(self):
        """(codes uint32[2 B], nmask uint32[B]): the packed planes as the device holds them."""
        n_blocks = int(((np.diff(self.seq_off) + 31) // 32).sum())
        codes = np.zeros(max(2 * n_blocks, 1), dtype=np.uint32)
        nmask = np.zeros(max(n_blocks, 1), dtype=np.uint32)
        with self.ctx._lock:
            check(self._lib.msb_seqs_to_packed(self.ctx._h, self._h, ctypes.c_void_p(codes.ctypes.data),
                                               ctypes.c_void_p(nmask.ctypes.data)))
        return codes[:2 * n_blocks], nmask[:n_blocks]

    def extract(self, src_idx, start, end):
        """A new sequence set cut out of this (resident) one on the device: sequence i = bases
        [start[i], end[i]) of sequence src_idx[i], `end` clipped at the source length like
        pysam's fetch (genome/__init__.py:135).  No sequence bytes cross PCIe."""
        src_idx = np.ascontiguousarray(np.asarray(src_idx, dtype=np.int32))
        start = np.ascontiguousarray(np.asarray(start, dtype=np.int64))
        end = np.ascontiguousarray(np.asarray(end, dtype=np.int64))
        if not (src_idx.shape == start.shape == end.shape and src_idx.ndim == 1):
            raise ValueError("src_idx, start and end must be 1-d arrays of one length")
        h = ctypes.c_void_p()
        with self.ctx._lock:
            check(self._lib.msb_seqs_extract(self.ctx._h, self._h, len(src_idx), ptr(src_idx, ctypes.c_int32),
                                             ptr(start, ctypes.c_int64), ptr(end, ctypes.c_int64), ctypes.byref(h)))
        return SequenceSet(self.ctx, _handle=h)

    def extract_subst(self, src_idx, start, end, sub_off, sub_pos, sub_code):
        """`extract` with bases substituted (msb_seqs_extract_subst): base sub_pos[k] of sequence i (relative to
        its start), k in [sub_off[i], sub_off[i + 1]), becomes the A/C/G/T code sub_code[k] (0..3).  Only the
        interval and substitution tables cross PCIe."""
        src_idx = np.ascontiguousarray(np.asarray(src_idx, dtype=np.int32))
        start = np.ascontiguousarray(np.asarray(start, dtype=np.int64))
        end = np.ascontiguousarray(np.asarray(end, dtype=np.int64))
        sub_off = np.ascontiguousarray(np.asarray(sub_off, dtype=np.int64))
        sub_pos = np.ascontiguousarray(np.asarray(sub_pos, dtype=np.int32))
        sub_code = np.ascontiguousarray(np.asarray(sub_code, dtype=np.uint8))
        if not (src_idx.shape == start.shape == end.shape and src_idx.ndim == 1):
            raise ValueError("src_idx, start and end must be 1-d arrays of one length")
        if sub_off.shape != (len(src_idx) + 1,) or sub_pos.shape != sub_code.shape or len(sub_pos) != int(sub_off[-1]):
            raise ValueError("sub_off must have n + 1 entries and sub_pos / sub_code sub_off[-1]")
        h = ctypes.c_void_p()
        with self.ctx._lock:
            check(self._lib.msb_seqs_extract_subst(self.ctx._h, self._h, len(src_idx), ptr(src_idx, ctypes.c_int32),
                                                   ptr(start, ctypes.c_int64), ptr(end, ctypes.c_int64),
                                                   ptr(sub_off, ctypes.c_int64), ptr(sub_pos, ctypes.c_int32),
                                                   ctypes.c_void_p(sub_code.ctypes.data), ctypes.byref(h)))
        return SequenceSet(self.ctx, _handle=h)

    def extract_splice(self, src_idx, start, end, splice_at, del_len, ins_off, ins_code):
        """`extract` with a splice (msb_seqs_extract_splice): bases [splice_at[i], splice_at[i] + del_len[i]) of
        sequence i (relative to its start) are replaced by the A/C/G/T codes ins_code[ins_off[i] .. ins_off[i + 1])
        (0..3); either side may be empty.  Only the interval and splice tables cross PCIe."""
        src_idx = np.ascontiguousarray(np.asarray(src_idx, dtype=np.int32))
        start = np.ascontiguousarray(np.asarray(start, dtype=np.int64))
        end = np.ascontiguousarray(np.asarray(end, dtype=np.int64))
        splice_at = np.ascontiguousarray(np.asarray(splice_at, dtype=np.int32))
        del_len = np.ascontiguousarray(np.asarray(del_len, dtype=np.int32))
        ins_off = np.ascontiguousarray(np.asarray(ins_off, dtype=np.int64))
        ins_code = np.ascontiguousarray(np.asarray(ins_code, dtype=np.uint8))
        if not (src_idx.shape == start.shape == end.shape == splice_at.shape == del_len.shape and src_idx.ndim == 1):
            raise ValueError("src_idx, start, end, splice_at and del_len must be 1-d arrays of one length")
        if ins_off.shape != (len(src_idx) + 1,) or ins_code.ndim != 1 or len(ins_code) != int(ins_off[-1]):
            raise ValueError("ins_off must have n + 1 entries and ins_code ins_off[-1]")
        h = ctypes.c_void_p()
        with self.ctx._lock:
            check(self._lib.msb_seqs_extract_splice(self.ctx._h, self._h, len(src_idx), ptr(src_idx, ctypes.c_int32),
                                                    ptr(start, ctypes.c_int64), ptr(end, ctypes.c_int64),
                                                    ptr(splice_at, ctypes.c_int32), ptr(del_len, ctypes.c_int32),
                                                    ptr(ins_off, ctypes.c_int64), ctypes.c_void_p(ins_code.ctypes.data),
                                                    ctypes.byref(h)))
        return SequenceSet(self.ctx, _handle=h)

    def extract_edits(self, src_idx, start, end, edit_off, edit_at, edit_del, ins_off, ins_code):
        """`extract` with several edits per sequence (msb_seqs_extract_edits): edit k in [edit_off[i], edit_off[i + 1])
        of sequence i replaces its bases [edit_at[k], edit_at[k] + edit_del[k]) (relative to the interval) by the A/C/G/T
        codes ins_code[ins_off[k] .. ins_off[k + 1]) (0..3).  The edits of a sequence are ordered and do not overlap.
        Only the interval and edit tables cross PCIe."""
        src_idx = np.ascontiguousarray(np.asarray(src_idx, dtype=np.int32))
        start = np.ascontiguousarray(np.asarray(start, dtype=np.int64))
        end = np.ascontiguousarray(np.asarray(end, dtype=np.int64))
        edit_off = np.ascontiguousarray(np.asarray(edit_off, dtype=np.int64))
        edit_at = np.ascontiguousarray(np.asarray(edit_at, dtype=np.int32))
        edit_del = np.ascontiguousarray(np.asarray(edit_del, dtype=np.int32))
        ins_off = np.ascontiguousarray(np.asarray(ins_off, dtype=np.int64))
        ins_code = np.ascontiguousarray(np.asarray(ins_code, dtype=np.uint8))
        if not (src_idx.shape == start.shape == end.shape and src_idx.ndim == 1):
            raise ValueError("src_idx, start and end must be 1-d arrays of one length")
        if edit_off.shape != (len(src_idx) + 1,) or edit_at.shape != edit_del.shape or edit_at.shape != (int(edit_off[-1]),):
            raise ValueError("edit_off must have n + 1 entries and edit_at / edit_del edit_off[-1]")
        if ins_off.shape != (len(edit_at) + 1,) or ins_code.ndim != 1 or len(ins_code) != int(ins_off[-1]):
            raise ValueError("ins_off must have one entry per edit + 1 and ins_code ins_off[-1]")
        h = ctypes.c_void_p()
        with self.ctx._lock:
            check(self._lib.msb_seqs_extract_edits(self.ctx._h, self._h, len(src_idx), ptr(src_idx, ctypes.c_int32),
                                                   ptr(start, ctypes.c_int64), ptr(end, ctypes.c_int64),
                                                   ptr(edit_off, ctypes.c_int64), ptr(edit_at, ctypes.c_int32),
                                                   ptr(edit_del, ctypes.c_int32), ptr(ins_off, ctypes.c_int64),
                                                   ctypes.c_void_p(ins_code.ctypes.data), ctypes.byref(h)))
        return SequenceSet(self.ctx, _handle=h)

    def window_ncount(self, src_idx, start, length):
        """Non-ACGT bases in each window [start[i], start[i] + length) of sequence src_idx[i]."""
        src_idx = np.ascontiguousarray(np.asarray(src_idx, dtype=np.int32))
        start = np.ascontiguousarray(np.asarray(start, dtype=np.int64))
        out = np.zeros(max(len(src_idx), 1), dtype=np.int32)
        with self.ctx._lock:
            check(self._lib.msb_seqs_window_ncount(self.ctx._h, self._h, len(src_idx), ptr(src_idx, ctypes.c_int32),
                                                   ptr(start, ctypes.c_int64), int(length), ptr(out, ctypes.c_int32)))
        return out[:len(src_idx)]

    def set_start_limit(self, limit):
        """Windows may only start at the first limit[i] positions of sequence i (chunked genome
        scans: starts inside the overlap belong to the next chunk).  None restores the default."""
        if limit is None:
            with self.ctx._lock:
                check(self._lib.msb_seqs_set_start_limit(self._h, None))
            return
        limit = np.ascontiguousarray(np.asarray(limit, dtype=np.int32))
        if limit.shape != (self.n,):
            raise ValueError("one start limit per sequence is required")
        with self.ctx._lock:
            check(self._lib.msb_seqs_set_start_limit(self._h, ptr(limit, ctypes.c_int32)))

    def codes(self):
        """Parity accessor: the reference's int8 codes (cscore.c:81-114) decoded from the device."""
        out = np.empty(max(self.total_bp, 1), dtype=np.int8)
        with self.ctx._lock:
            check(self._lib.msb_seqs_codes(self.ctx._h, self._h, ptr(out, ctypes.c_int8)))
        return out[:self.total_bp]

    def close(self):
        if self._h:
            self._lib.msb_seqs_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ScanResult:
    """Sites of one scan in the reference's order (motif-major; sequence, start ascending;
    forward before reverse).  Arrays are views into pinned memory owned by the result.  A result of
    an asynchronous scan (`async_=True`) knows `n_sites` at once; everything else waits for the
    device-to-host copy on first use (`wait()`)."""

    def __init__(self, ctx, handle, n_motifs):
        self.ctx = ctx
        self._lib = ctx._lib
        self._h = handle
        self.n_motifs = n_motifs
        n = ctypes.c_int64(0)
        check(self._lib.msb_result_total(self._h, ctypes.byref(n)))
        self.n_sites = n.value
        self._loaded = False

    def wait(self):
        """Block until the copies have landed; `counts` / `offsets` are valid afterwards.  The site arrays are
        bound on first use (`seq_idx`, `start`, `score`, `strand`): for a compact result that first use
        decodes the positions on the host, which a caller that gathers with `merge_sites_compact` never pays."""
        if self._loaded:
            return self
        n_motifs = self.n_motifs
        counts = np.zeros(max(n_motifs, 1), dtype=np.int64)
        check(self._lib.msb_result_counts(self._h, ptr(counts, ctypes.c_int64)))   # waits for the copies
        self.counts = counts[:n_motifs]
        self.offsets = np.zeros(n_motifs + 1, dtype=np.int64)
        np.cumsum(self.counts, out=self.offsets[1:])
        self._loaded = True
        return self

    def _bind_arrays(self):
        self.wait()
        p_seq, p_start = _lib.c_i32p(), _lib.c_i32p()
        p_score, p_strand = _lib.c_f64p(), _lib.c_i8p()
        check(self._lib.msb_result_arrays(self._h, ctypes.byref(p_seq), ctypes.byref(p_start),
                                          ctypes.byref(p_score), ctypes.byref(p_strand)))
        if self.n_sites:
            shape = (self.n_sites,)
            self.seq_idx = np.ctypeslib.as_array(p_seq, shape=shape)
            self.start = np.ctypeslib.as_array(p_start, shape=shape)
            self.score = np.ctypeslib.as_array(p_score, shape=shape)
            self.strand = np.ctypeslib.as_array(p_strand, shape=shape)
        else:
            self.seq_idx = np.zeros(0, dtype=np.int32)
            self.start = np.zeros(0, dtype=np.int32)
            self.score = np.zeros(0, dtype=np.float64)
            self.strand = np.zeros(0, dtype=np.int8)

    def __getattr__(self, name):
        if name in ("counts", "offsets") and not self.__dict__.get("_loaded", True):
            self.wait()
            return self.__dict__[name]
        if name in ("seq_idx", "start", "score", "strand") and "_h" in self.__dict__ and "seq_idx" not in self.__dict__:
            self._bind_arrays()
            return self.__dict__[name]
        raise AttributeError(name)

    def compact(self):
        """The raw arrays of a compact result (`compact=True` scans): (pos_strand uint32[n], score float64[n],
        poff int64[n_seqs + 1]) -- see msb_result_compact -- or None when the result is an ordinary one."""
        ps, sc, po = ctypes.POINTER(ctypes.c_uint32)(), _lib.c_f64p(), _lib.c_i64p()
        ns = ctypes.c_int64(0)
        check(self._lib.msb_result_compact(self._h, ctypes.byref(ps), ctypes.byref(sc), ctypes.byref(po), ctypes.byref(ns)))
        if not ps or self.n_sites == 0:
            return None
        return (np.ctypeslib.as_array(ps, shape=(self.n_sites,)), np.ctypeslib.as_array(sc, shape=(self.n_sites,)),
                np.ctypeslib.as_array(po, shape=(ns.value + 1,)))

    def detach(self):
        """Copy the arrays out of the pinned block and release it."""
        self.wait()
        self.seq_idx = self.seq_idx.copy()
        self.start = self.start.copy()
        self.score = self.score.copy()
        self.strand = self.strand.copy()
        self.close()
        return self

    def close(self):
        if self._h:
            self._lib.msb_result_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _flags(remove_dup=False, counts_only=False, async_=False, compact=False):
    return ((_lib.MSB_SCAN_DEDUP if remove_dup else 0) | (_lib.MSB_SCAN_COUNTS if counts_only else 0)
            | (_lib.MSB_SCAN_ASYNC if async_ else 0) | (_lib.MSB_SCAN_COMPACT if compact else 0))


def merge_motif_major(counts, arrays, add=None, n_threads=None):
    """Gather motif-major arrays of several scans (one per GPU or batch, parts in ascending sequence
    order) into one motif-major array (msb_merge_motif_major: host memcpy on several threads, no
    sort, no pickling).  `counts` int64[n_parts, n_motifs]; `arrays` one array per part; `add`
    optional per-part addend for int32 arrays (the part's first global sequence index)."""
    import os
    counts = np.ascontiguousarray(np.asarray(counts, dtype=np.int64))
    n_parts, n_motifs = counts.shape
    if n_parts == 0:
        return np.zeros(0, dtype=np.int32)
    dtype = arrays[0].dtype
    keep = [np.ascontiguousarray(a) for a in arrays]
    src = (ctypes.c_void_p * n_parts)(*[ctypes.c_void_p(a.ctypes.data if a.size else 0) for a in keep])
    out = np.empty(int(counts.sum()), dtype=dtype)
    add_arr = None if add is None else np.ascontiguousarray(np.asarray(add, dtype=np.int64))
    check(_lib.load().msb_merge_motif_major(n_parts, n_motifs, ptr(counts, ctypes.c_int64), src,
                                            ctypes.c_void_p(out.ctypes.data if out.size else 0), dtype.itemsize,
                                            ptr(add_arr, ctypes.c_int64) if add_arr is not None else None,
                                            int(n_threads or min(os.cpu_count() or 1, 16))))
    return out


def scan(ctx, motifs, seqs, strand, remove_dup=False, async_=False, compact=False):
    """Scan; with remove_dup the reference's adjacent-site de-duplication (scanner.py:156-193)
    runs on the device before the sites are copied back.  `async_`: return while the copy of the
    sites is still in flight (the next scan on `ctx` overlaps it; `ScanResult.wait`)."""
    h = ctypes.c_void_p()
    flags = _flags(remove_dup, async_=async_, compact=compact)
    with ctx._lock:
        check(ctx._lib.msb_scan_ex(ctx._h, motifs._h, seqs._h, int(strand), flags, ctypes.byref(h)))
    return ScanResult(ctx, h, motifs.n)


def scan_ascii(ctx, motifs, blob, seq_off, strand, remove_dup=False, async_=False):
    """Host ASCII in, host sites out in one call (msb_scan_ascii): the upload of the sequence bytes
    is cut into slices that overlap with the scan.  `blob` should live in pinned memory
    (`pinned_array`) for the overlap to happen; any uint8 array works."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8) if not isinstance(blob, np.ndarray) else blob
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    h = ctypes.c_void_p()
    flags = _flags(remove_dup, async_=async_)
    data = blob.ctypes.data if blob.size else None
    with ctx._lock:
        check(ctx._lib.msb_scan_ascii(ctx._h, motifs._h, len(seq_off) - 1, ctypes.c_void_p(data), ptr(seq_off, ctypes.c_int64),
                                      int(strand), flags, None, ctypes.byref(h)))
    return ScanResult(ctx, h, motifs.n)


def merge_sites(counts, seq_idx, start, score, strand, seq_to_group=None, seq_offset=None, n_threads=None):
    """Gather the site lists of several scans (parts in ascending sequence order) into one motif-major list in
    ONE pass over the data (msb_merge_sites), translating each part's local sequence numbers: sequence q of
    part p becomes `seq_to_group[p][q]` and its starts move by `seq_offset[p][q]`.  Returns
    (group int32, start int32, score float64, strand int8)."""
    import os
    counts = np.ascontiguousarray(np.asarray(counts, dtype=np.int64))
    n_parts, n_motifs = counts.shape
    total = int(counts.sum())
    out = (np.empty(total, np.int32), np.empty(total, np.int32), np.empty(total, np.float64), np.empty(total, np.int8))
    if n_parts == 0 or total == 0:
        return out

    def table(arrays, dtype):
        if arrays is None:
            return None, None
        keep = [np.ascontiguousarray(a, dtype=dtype) for a in arrays]
        return keep, (ctypes.c_void_p * n_parts)(*[ctypes.c_void_p(a.ctypes.data if a.size else 0) for a in keep])
    keep = [table(seq_idx, np.int32), table(start, np.int32), table(score, np.float64), table(strand, np.int8),
            table(seq_to_group, np.int32), table(seq_offset, np.int32)]
    check(_lib.load().msb_merge_sites(n_parts, n_motifs, ptr(counts, ctypes.c_int64), *[k[1] for k in keep],
                                      *[ctypes.c_void_p(o.ctypes.data) for o in out],
                                      int(n_threads or min(os.cpu_count() or 1, 16))))
    return out


def merge_sites_compact(counts, results, seq_to_group=None, seq_offset=None, n_threads=None):
    """`merge_sites` straight from compact results (`ScanResult.compact()` of every part): the owning sequence
    of a site is found while it is copied."""
    import os
    counts = np.ascontiguousarray(np.asarray(counts, dtype=np.int64))
    n_parts, n_motifs = counts.shape
    total = int(counts.sum())
    out = (np.empty(total, np.int32), np.empty(total, np.int32), np.empty(total, np.float64), np.empty(total, np.int8))
    if n_parts == 0 or total == 0:
        return out
    raw = [r.compact() for r in results]

    def table(arrays, dtype):
        if arrays is None:
            return None, None
        keep = [np.ascontiguousarray(a, dtype=dtype) for a in arrays]
        return keep, (ctypes.c_void_p * n_parts)(*[ctypes.c_void_p(a.ctypes.data if a.size else 0) for a in keep])
    empty = (np.zeros(1, np.uint32), np.zeros(1, np.float64), np.zeros(2, np.int64))
    raw = [x if x is not None else empty for x in raw]
    keep = [table([x[0] for x in raw], np.uint32), table([x[1] for x in raw], np.float64), table([x[2] for x in raw], np.int64),
            table(seq_to_group, np.int32), table(seq_offset, np.int32)]
    n_seqs = np.array([len(x[2]) - 1 for x in raw], dtype=np.int64)
    check(_lib.load().msb_merge_sites_compact(n_parts, n_motifs, ptr(counts, ctypes.c_int64), keep[0][1], keep[1][1], keep[2][1],
                                              ptr(n_seqs, ctypes.c_int64), keep[3][1], keep[4][1],
                                              *[ctypes.c_void_p(o.ctypes.data) for o in out],
                                              int(n_threads or min(os.cpu_count() or 1, 16))))
    return out


class PinnedArray:
    """A uint8 numpy view of page-locked host memory (msb_pinned_alloc); `.array` is the view."""

    def __init__(self, nbytes):
        self._lib = _lib.load()
        self._p = ctypes.c_void_p()
        check(self._lib.msb_pinned_alloc(int(nbytes), ctypes.byref(self._p)))
        self.array = np.ctypeslib.as_array(ctypes.cast(self._p, ctypes.POINTER(ctypes.c_uint8)), shape=(max(int(nbytes), 1),))[:int(nbytes)]

    def close(self):
        if self._p:
            self._lib.msb_pinned_free(self._p)
            self._p = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scan_device(ctx, motifs, seqs, strand, remove_dup=False, counts_only=False):
    """Kernels only (results stay on the device); returns the number of sites.  `counts_only`: the
    sites are not even ordered -- `ctx.site_counts` is all that can be read afterwards."""
    n = ctypes.c_int64(0)
    flags = _flags(remove_dup, counts_only)
    with ctx._lock:
        check(ctx._lib.msb_scan_device(ctx._h, motifs._h, seqs._h, int(strand), flags, ctypes.byref(n)))
    return n.value


def _ranges(ranges):
    r = np.ascontiguousarray(np.asarray(ranges, dtype=np.int64).reshape(-1, 3))
    return (len(r), np.ascontiguousarray(r[:, 0]), np.ascontiguousarray(r[:, 1]), np.ascontiguousarray(r[:, 2]))


def scan_ranges(ctx, motifs, seqs, strand, ranges, async_=False, compact=False, remove_dup=False):
    """Scan only the windows that start in the given (sequence index, start, end) ranges of a
    resident sequence set; sites refer to the sequences of `seqs` (msb_scan_ranges).  `remove_dup`:
    de-duplicate per range (scanner.py:171-193), which needs at most one range per sequence; the chains
    at the range edges can then be read with `ctx.boundary_sites()`."""
    n, a, b, c = _ranges(ranges)
    h = ctypes.c_void_p()
    flags = _flags(remove_dup, async_=async_, compact=compact)
    with ctx._lock:
        check(ctx._lib.msb_scan_ranges(ctx._h, motifs._h, seqs._h, int(strand), flags, n, ptr(a, ctypes.c_int64),
                                       ptr(b, ctypes.c_int64), ptr(c, ctypes.c_int64), ctypes.byref(h)))
    return ScanResult(ctx, h, motifs.n)


def scan_ranges_device(ctx, motifs, seqs, strand, ranges, counts_only=False, remove_dup=False):
    """The same, results left on the device (`ctx.site_counts`, `ctx.cell_stats`); returns the number of sites."""
    n, a, b, c = _ranges(ranges)
    total = ctypes.c_int64(0)
    flags = _flags(remove_dup, counts_only)
    with ctx._lock:
        check(ctx._lib.msb_scan_ranges_device(ctx._h, motifs._h, seqs._h, int(strand), flags, n, ptr(a, ctypes.c_int64),
                                              ptr(b, ctypes.c_int64), ptr(c, ctypes.c_int64), ctypes.byref(total)))
    return total.value


def scan_variants(ctx, motifs, ref, alt, core_start, core_len, strand):
    """Variant-effect scan (msb_scan_variants): sequence i of `ref` / `alt` is allele i's context without / with the
    allele, its changed bases [core_start[i], core_start[i] + core_len[i]).  Returns a dict of row arrays in (allele,
    motif, start, strand) order: allele int32, motif int32, start int32 (relative to the context), strand int8 (1 / 2),
    ref_score / alt_score float64 (the window's exact score on each allele) and effect int8 (1 loss, 2 gain, 3 both)."""
    core_start = np.ascontiguousarray(np.asarray(core_start, dtype=np.int32))
    core_len = np.ascontiguousarray(np.asarray(core_len, dtype=np.int32))
    if core_start.shape != (ref.n,) or core_len.shape != (ref.n,):
        raise ValueError("one core per context is required")
    with ctx._lock:
        n = ctypes.c_int64(0)
        check(ctx._lib.msb_scan_variants(ctx._h, motifs._h, ref._h, alt._h, ptr(core_start, ctypes.c_int32),
                                         ptr(core_len, ctypes.c_int32), int(strand), ctypes.byref(n)))
        return _variant_rows(ctx, n.value)


def scan_variants_ex(ctx, motifs, ref, alt, core_start, ref_core_len, alt_core_len, strand):
    """scan_variants with a changed length per side (msb_scan_variants_ex, indels): the changed bases are
    [core_start[i], core_start[i] + ref_core_len[i]) of ref context i and [core_start[i], core_start[i] +
    alt_core_len[i]) of alt context i.  The same row arrays; effect 5 is a loss and 6 a gain whose window does not
    exist on the other allele (its score NaN)."""
    core_start = np.ascontiguousarray(np.asarray(core_start, dtype=np.int32))
    ref_core_len = np.ascontiguousarray(np.asarray(ref_core_len, dtype=np.int32))
    alt_core_len = np.ascontiguousarray(np.asarray(alt_core_len, dtype=np.int32))
    if not core_start.shape == ref_core_len.shape == alt_core_len.shape == (ref.n,):
        raise ValueError("one core per context is required")
    with ctx._lock:
        n = ctypes.c_int64(0)
        check(ctx._lib.msb_scan_variants_ex(ctx._h, motifs._h, ref._h, alt._h, ptr(core_start, ctypes.c_int32),
                                            ptr(ref_core_len, ctypes.c_int32), ptr(alt_core_len, ctypes.c_int32),
                                            int(strand), ctypes.byref(n)))
        return _variant_rows(ctx, n.value)


def scan_haplotypes(ctx, motifs, ref, alt, edit_off, edit_at, edit_ref_len, edit_alt_len, strand):
    """scan_variants_ex with several edits per context (msb_scan_haplotypes): edit k in [edit_off[i], edit_off[i + 1])
    of context i replaces the ref bases [edit_at[k], edit_at[k] + edit_ref_len[k]) by edit_alt_len[k] alt bases.  The
    same row arrays with `context` for `allele`, `start` on the row's own side (alt for effect 2 / 6, else ref) and
    `other_start`, the window's start on the other side (-1: none); rows in (context, motif, start, strand, ref before
    alt) order."""
    edit_off = np.ascontiguousarray(np.asarray(edit_off, dtype=np.int64))
    edit_at = np.ascontiguousarray(np.asarray(edit_at, dtype=np.int32))
    edit_ref_len = np.ascontiguousarray(np.asarray(edit_ref_len, dtype=np.int32))
    edit_alt_len = np.ascontiguousarray(np.asarray(edit_alt_len, dtype=np.int32))
    if edit_off.shape != (ref.n + 1,):
        raise ValueError("edit_off must have one entry per context + 1")
    if not edit_at.shape == edit_ref_len.shape == edit_alt_len.shape == (int(edit_off[-1]),):
        raise ValueError("edit_at / edit_ref_len / edit_alt_len must have edit_off[-1] entries")
    with ctx._lock:
        n = ctypes.c_int64(0)
        check(ctx._lib.msb_scan_haplotypes(ctx._h, motifs._h, ref._h, alt._h, ptr(edit_off, ctypes.c_int64),
                                           ptr(edit_at, ctypes.c_int32), ptr(edit_ref_len, ctypes.c_int32),
                                           ptr(edit_alt_len, ctypes.c_int32), int(strand), ctypes.byref(n)))
        out = _variant_rows(ctx, n.value, other=True)
    out["context"] = out.pop("allele")
    return out


def _variant_rows(ctx, k, other=False):
    """The k rows of the last variant scan on `ctx` (caller holds its lock); `other`: with other_start."""
    n = ctypes.c_int64(0)
    out = dict(allele=np.zeros(k, np.int32), motif=np.zeros(k, np.int32), start=np.zeros(k, np.int32),
               strand=np.zeros(k, np.int8), ref_score=np.zeros(k, np.float64), alt_score=np.zeros(k, np.float64),
               effect=np.zeros(k, np.int8))
    if other:
        out["other_start"] = np.zeros(k, np.int32)
    if k:
        args = [ctx._h, k, ctypes.byref(n), ptr(out["allele"], ctypes.c_int32), ptr(out["motif"], ctypes.c_int32),
                ptr(out["start"], ctypes.c_int32), ptr(out["strand"], ctypes.c_int8), ptr(out["ref_score"], ctypes.c_double),
                ptr(out["alt_score"], ctypes.c_double), ptr(out["effect"], ctypes.c_int8)]
        if other:
            check(ctx._lib.msb_scan_device_haplotype_rows(*args, ptr(out["other_start"], ctypes.c_int32)))
        else:
            check(ctx._lib.msb_scan_device_variant_rows(*args))
    return out


def score(ctx, motifs, seqs, strand):
    out = np.empty((motifs.n, seqs.n), dtype=np.float64)
    buf = out if out.size else np.zeros(1, dtype=np.float64)
    with ctx._lock:
        check(ctx._lib.msb_score(ctx._h, motifs._h, seqs._h, int(strand), ptr(buf, ctypes.c_double)))
    return out


def score_select(ctx, motifs, seqs, strand, ranks):
    ranks = np.ascontiguousarray(np.asarray(ranks, dtype=np.int64))
    out = np.empty((motifs.n, len(ranks)), dtype=np.float64)
    buf = out if out.size else np.zeros(1, dtype=np.float64)
    with ctx._lock:
        check(ctx._lib.msb_score_select(ctx._h, motifs._h, seqs._h, int(strand), len(ranks),
                                        ptr(ranks, ctypes.c_int64), ptr(buf, ctypes.c_double)))
    return out
