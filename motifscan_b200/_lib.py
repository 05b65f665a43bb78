"""ctypes binding of libmsb200.so (C ABI: include/msb200.h).

The library is the only implementation of the scan path in this package: if it is missing, or no
CUDA device is usable, calls raise -- there is no CPU fallback.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MSB200_LIB: an experiment build of the same library (motifscan_b200.build(out=..., defines=...))
LIB_PATH = os.environ.get("MSB200_LIB") or os.path.join(_HERE, "libmsb200.so")

MSB_OK, MSB_EINVAL, MSB_ENOMEM, MSB_ECUDA, MSB_ESHORT = 0, -1, -2, -3, -4
MSB_SCAN_DEDUP = 1
MSB_SCAN_COUNTS = 2
MSB_SCAN_ASYNC = 4
MSB_SCAN_COMPACT = 8
MSB_SEQS_ASYNC = 1
CENTRALITY_MAX_CELLS = 1 << 26    # MSB_CENTRALITY_MAX_CELLS
T_NAMES = ("h2d", "encode", "prefilter", "exact", "order", "d2h", "score", "select", "rows", "row_sort", "pairs", "spacing",
           "centrality")
C_NAMES = ("candidates", "dirty", "hits", "launches", "retries", "prefilter_launches")

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_i8p = ctypes.POINTER(ctypes.c_int8)
c_vp = ctypes.c_void_p

# name -> (restype, argtypes); one entry per symbol declared in include/msb200.h
SIGNATURES = {
    "msb_last_error": (ctypes.c_char_p, []),
    "msb_version": (ctypes.c_int, []),
    "msb_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "msb_device_pci_bus_id": (ctypes.c_int, [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]),
    "msb_ctx_create": (ctypes.c_int, [ctypes.c_int, c_vp, ctypes.POINTER(c_vp)]),
    "msb_ctx_destroy": (ctypes.c_int, [c_vp]),
    "msb_ctx_sync": (ctypes.c_int, [c_vp]),
    "msb_ctx_timings": (ctypes.c_int, [c_vp, c_f64p, ctypes.c_int]),
    "msb_ctx_counters": (ctypes.c_int, [c_vp, c_i64p, ctypes.c_int]),
    "msb_ctx_set_option": (ctypes.c_int, [c_vp, ctypes.c_char_p, ctypes.c_int]),
    "msb_pinned_alloc": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(c_vp)]),
    "msb_pinned_free": (ctypes.c_int, [c_vp]),
    "msb_motifs_create": (ctypes.c_int, [c_vp, ctypes.c_int32, c_i32p, c_f64p, c_i64p, c_f64p,
                                         ctypes.POINTER(c_vp)]),
    "msb_motifs_set_cutoffs": (ctypes.c_int, [c_vp, c_f64p]),
    "msb_motifs_count": (ctypes.c_int, [c_vp, c_i32p]),
    "msb_motifs_max_raw": (ctypes.c_int, [c_vp, c_f64p]),
    "msb_motifs_destroy": (ctypes.c_int, [c_vp]),
    "msb_seqs_from_ascii": (ctypes.c_int, [c_vp, ctypes.c_int64, c_vp, c_i64p, ctypes.POINTER(c_vp)]),
    "msb_seqs_from_packed": (ctypes.c_int, [c_vp, ctypes.c_int64, c_i64p, c_vp, c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "msb_seqs_wait": (ctypes.c_int, [c_vp]),
    "msb_seqs_to_packed": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp]),
    "msb_seqs_extract": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, c_i64p, c_i64p, ctypes.POINTER(c_vp)]),
    "msb_seqs_extract_subst": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, c_i64p, c_i64p, c_i64p, c_i32p, c_vp,
                                              ctypes.POINTER(c_vp)]),
    "msb_seqs_extract_splice": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, c_i64p, c_i64p, c_i32p, c_i32p, c_i64p, c_vp,
                                               ctypes.POINTER(c_vp)]),
    "msb_seqs_extract_edits": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, c_i64p, c_i64p, c_i64p, c_i32p, c_i32p, c_i64p,
                                              c_vp, ctypes.POINTER(c_vp)]),
    "msb_seqs_lengths": (ctypes.c_int, [c_vp, c_i64p]),
    "msb_seqs_window_ncount": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, c_i64p, ctypes.c_int32, c_i32p]),
    "msb_seqs_set_start_limit": (ctypes.c_int, [c_vp, c_i32p]),
    "msb_seqs_count": (ctypes.c_int, [c_vp, c_i64p, c_i64p]),
    "msb_seqs_codes": (ctypes.c_int, [c_vp, c_vp, c_i8p]),
    "msb_seqs_destroy": (ctypes.c_int, [c_vp]),
    "msb_scan": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "msb_scan_ex": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "msb_scan_ascii": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp, c_i64p, ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(c_vp), ctypes.POINTER(c_vp)]),
    "msb_scan_ranges": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64, c_i64p, c_i64p,
                                       c_i64p, ctypes.POINTER(c_vp)]),
    "msb_scan_ranges_device": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64, c_i64p,
                                              c_i64p, c_i64p, c_i64p]),
    "msb_scan_device": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_i64p]),
    "msb_scan_device_counts": (ctypes.c_int, [c_vp, c_i64p, ctypes.c_int32]),
    "msb_scan_device_region_counts": (ctypes.c_int, [c_vp, c_i64p, ctypes.c_int32]),
    "msb_scan_device_boundary_sites": (ctypes.c_int, [c_vp, ctypes.c_int64, c_i64p, c_i32p, c_i32p, c_i32p, c_f64p, c_i8p, c_i8p]),
    "msb_scan_device_cell_stats": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int64, c_i64p, c_f64p]),
    "msb_scan_device_pair_counts": (ctypes.c_int, [c_vp, ctypes.c_int32, ctypes.c_int64, c_i64p]),
    "msb_scan_device_spacing": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int32, c_i32p, ctypes.c_int32, c_i64p]),
    "msb_scan_device_centrality": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_i32p, ctypes.c_int32, ctypes.c_int32, c_i64p,
                                                  c_i64p]),
    "msb_scan_variants": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32p, c_i32p, ctypes.c_int, c_i64p]),
    "msb_scan_variants_ex": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32p, c_i32p, c_i32p, ctypes.c_int, c_i64p]),
    "msb_scan_device_variant_rows": (ctypes.c_int, [c_vp, ctypes.c_int64, c_i64p, c_i32p, c_i32p, c_i32p, c_i8p, c_f64p, c_f64p,
                                                    c_i8p]),
    "msb_scan_haplotypes": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64p, c_i32p, c_i32p, c_i32p, ctypes.c_int, c_i64p]),
    "msb_scan_device_haplotype_rows": (ctypes.c_int, [c_vp, ctypes.c_int64, c_i64p, c_i32p, c_i32p, c_i32p, c_i8p, c_f64p,
                                                      c_f64p, c_i8p, c_i32p]),
    "msb_result_wait": (ctypes.c_int, [c_vp]),
    "msb_merge_motif_major": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, c_i64p, ctypes.POINTER(c_vp), c_vp,
                                             ctypes.c_int32, c_i64p, ctypes.c_int32]),
    "msb_merge_sites": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, c_i64p] + [ctypes.POINTER(c_vp)] * 6 +
                        [c_vp, c_vp, c_vp, c_vp, ctypes.c_int32]),
    "msb_merge_sites_compact": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, c_i64p] + [ctypes.POINTER(c_vp)] * 3 + [c_i64p] +
                                [ctypes.POINTER(c_vp)] * 2 + [c_vp, c_vp, c_vp, c_vp, ctypes.c_int32]),
    "msb_result_compact": (ctypes.c_int, [c_vp, ctypes.POINTER(ctypes.POINTER(ctypes.c_uint32)), ctypes.POINTER(c_f64p),
                                          ctypes.POINTER(c_i64p), c_i64p]),
    "msb_format_site_tables": (ctypes.c_int, [ctypes.c_int32, c_i64p, c_i32p, c_f64p, ctypes.c_int64, ctypes.c_int64, ctypes.c_char_p,
                                              c_i64p, ctypes.POINTER(c_vp), c_i64p, ctypes.POINTER(c_vp), c_i64p, ctypes.c_int32]),
    "msb_format_cell_tables": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, c_i64p, c_f64p, ctypes.c_char_p, c_i64p,
                                              ctypes.POINTER(c_vp), c_i64p, ctypes.POINTER(c_vp), c_i64p, ctypes.c_int32]),
    "msb_write_sites_bed": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int64, c_i32p, c_i32p, c_i64p, c_f64p, c_i8p, ctypes.c_int32,
                                           ctypes.c_int64, ctypes.c_char_p, c_i64p, ctypes.c_int32]),
    "msb_write_variant_table": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int64, c_i32p, c_i32p, c_i32p, c_i8p,
                                               c_f64p, c_f64p, c_i8p, ctypes.c_int64, ctypes.c_char_p, c_i64p, ctypes.c_int32,
                                               ctypes.c_char_p, c_i64p, c_i32p, ctypes.c_int32]),
    "msb_write_haplotype_table": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int64, c_i32p, c_i32p, c_i64p,
                                                 c_i64p, c_i8p, c_f64p, c_f64p, c_i8p, ctypes.c_int64, ctypes.c_char_p, c_i64p,
                                                 ctypes.c_int32, ctypes.c_char_p, c_i64p, c_i32p, ctypes.c_int32]),
    "msb_write_cooccur_table": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int64, c_i32p, c_i32p, ctypes.c_int32,
                                               ctypes.c_char_p, c_i64p, c_i64p, c_i64p, c_f64p, c_f64p, c_f64p, c_f64p, c_f64p,
                                               c_i64p, c_f64p, c_f64p, c_f64p, c_f64p, ctypes.c_int32]),
    "msb_text_free": (ctypes.c_int, [c_vp]),
    "msb_result_total": (ctypes.c_int, [c_vp, c_i64p]),
    "msb_result_counts": (ctypes.c_int, [c_vp, c_i64p]),
    "msb_result_arrays": (ctypes.c_int, [c_vp, ctypes.POINTER(c_i32p), ctypes.POINTER(c_i32p),
                                         ctypes.POINTER(c_f64p), ctypes.POINTER(c_i8p)]),
    "msb_result_destroy": (ctypes.c_int, [c_vp]),
    "msb_score": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, c_f64p]),
    "msb_score_select": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int32, c_i64p, c_f64p]),
    "msb_c_scan_motif": (ctypes.c_int, [ctypes.c_int, ctypes.c_int32, c_i32p, c_f64p, c_i64p, c_f64p,
                                        ctypes.c_int64, c_vp, c_i64p, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "msb_c_score": (ctypes.c_int, [ctypes.c_int, ctypes.c_int32, c_i32p, c_f64p, c_i64p, ctypes.c_int64,
                                   c_vp, c_i64p, ctypes.c_int, c_f64p]),
}

_lib = None


class MsbError(RuntimeError):
    pass


def load():
    """Load libmsb200.so; raises if it has not been built (python -m motifscan_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MsbError(f"{LIB_PATH} not found: build it with `python -m motifscan_b200.build` "
                           "(there is no CPU fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc == MSB_OK:
        return
    msg = (load().msb_last_error() or b"").decode("utf-8", "replace")
    if rc == MSB_EINVAL or rc == MSB_ESHORT:
        raise ValueError(msg)
    if rc == MSB_ENOMEM:
        raise MemoryError(msg)
    raise MsbError(msg)


def ptr(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def device_count():
    n = ctypes.c_int(0)
    check(load().msb_device_count(ctypes.byref(n)))
    return n.value


def bind_thread_near(device):
    """Pin the calling host thread to the cores that are NUMA-local to a GPU (its PCI device's
    `local_cpulist`), so that the pinned buffers it allocates next and its copies stay on that GPU's side
    of the host.  Returns the core list, or None when the topology cannot be read (nothing is changed)."""
    try:
        buf = ctypes.create_string_buffer(32)
        check(load().msb_device_pci_bus_id(int(device), buf, 32))
        path = f"/sys/bus/pci/devices/{buf.value.decode().lower()}/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)        # pid 0 = the calling thread
        return sorted(cpus)
    except Exception:
        return None


def flatten_pwms(pwms):
    """Sequence of 4 x L_m matrices (lists or arrays; ints accepted like PyFloat_AsDouble does,
    cscore.c:65) -> (lens int32[n], mats float64[sum 4 L_m], mat_off int64[n])."""
    n = len(pwms)
    lens = np.empty(n, dtype=np.int32)
    mat_off = np.empty(n, dtype=np.int64)
    chunks = []
    at = 0
    for m, p in enumerate(pwms):
        a = np.ascontiguousarray(np.asarray(p, dtype=np.float64))
        if a.ndim != 2 or a.shape[0] != 4:
            raise ValueError(f"PWM {m}: expected a 4 x L matrix, got shape {a.shape}")
        lens[m] = a.shape[1]
        mat_off[m] = at
        at += a.size
        chunks.append(a.ravel())
    mats = np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.float64)
    if mats.size == 0:
        mats = np.zeros(1, dtype=np.float64)
    return lens, mats, mat_off


def flatten_seqs(seqs):
    """Sequence of str / bytes -> (uint8 array, seq_off int64[n+1]).  str is encoded as UTF-8,
    which is what the reference reads (PyUnicode_AsUTF8AndSize, cscore.c:83)."""
    bs = [s.encode("utf-8") if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        np.cumsum([len(b) for b in bs], out=off[1:])
    blob = np.frombuffer(b"".join(bs), dtype=np.uint8)
    return blob, off
