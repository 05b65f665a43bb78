/*
 * msb200.h -- C ABI of libmsb200.so, the B200 (sm_100a) implementation of MotifScan's
 * motif-scanning hot path.
 *
 * The reference exposes this path as a CPython extension module, `motifscan.motif.cscore`
 * (reference motifscan/motif/cscore.c:479-494), with two methods:
 *     c_scan_motif(pwms, cutoffs, seqs, strand, n_threads)   cscore.c:399-476
 *     c_score(pwms, seqs, strand, n_threads)                 cscore.c:231-302
 * called from motifscan/scanner.py:125 and motifscan/cli/motif.py:134.  This header is what a
 * binding for that module binds instead (see INTEGRATION.md for the ctypes stub): plain
 * pointers and sizes, no Python and no torch types.
 *
 * Conventions
 *   - every function returns MSB_OK (0) or a negative MSB_E* code; msb_last_error() returns a
 *     thread-local message for the last failure on the calling thread.  Nothing calls exit()
 *     (the reference does on hit-allocation failure, cscore.c:360-363).
 *   - the library keeps no global mutable state: all state, including every tuning option, hangs
 *     off an msb_ctx (one device, one stream).  Different contexts may be used from different
 *     host threads concurrently -- that is how one process drives several GPUs -- while calls on
 *     ONE context must be serialised by the caller (the reference's file-scope globals,
 *     cscore.c:26-34, make it single-caller).  The handle-less mirrors msb_c_scan_motif /
 *     msb_c_score keep one context per (calling thread, device) in thread-local storage.
 *   - PWMs are passed flat: motif m is the row-major 4 x lens[m] block at mats + mat_off[m]
 *     (rows A, C, G, T -- the reference's `double *matrix[4]`, cscore.c:6-11).
 *   - sequences are passed flat: sequence i is the ASCII bytes seq_bytes[seq_off[i] ..
 *     seq_off[i+1]).  Encoding follows cscore.c:81-114: A/a C/c G/g T/t -> 0..3, any other
 *     byte is "N" (contributes 0 to a score, cscore.c:346).
 *   - strand: 1 forward, 2 reverse, 3 both (cscore.c:176-177).
 *   - n_threads of the reference API has no equivalent here and is dropped.
 */
#ifndef MSB200_H
#define MSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSB_OK 0
#define MSB_EINVAL -1   /* bad argument (the reference performs no validation, cscore.c:117-120) */
#define MSB_ENOMEM -2   /* host or device allocation failed (reference: MemoryError / exit(1)) */
#define MSB_ECUDA -3    /* CUDA runtime error, no usable device, or kernel image mismatch */
#define MSB_ESHORT -4   /* c_score: a sequence is shorter than the longest motif (reference: UB) */

typedef struct msb_ctx msb_ctx;       /* one device + one stream + reusable scratch */
typedef struct msb_motifs msb_motifs; /* device-resident motif set: fp64 PWMs, cutoffs, tables */
typedef struct msb_seqs msb_seqs;     /* device-resident sequence set: 2-bit codes + N mask */
typedef struct msb_result msb_result; /* host-resident sites of one scan, reference order */

const char *msb_last_error(void);
int msb_version(void);
int msb_device_count(int *count);
/* PCI bus id of a device ("0000:1b:00.0"): hosts use it to find the GPU's NUMA-local cores
 * (/sys/bus/pci/devices/<id>/local_cpulist) before they allocate pinned buffers for it. */
int msb_device_pci_bus_id(int device, char *out, int len);

/* ---- context ------------------------------------------------------------------------------ */
/* `stream` is an optional cudaStream_t (as void*) to launch on, e.g. torch's current stream;
 * NULL makes the context create and own a non-blocking stream. */
int msb_ctx_create(int device, void *stream, msb_ctx **ctx);
int msb_ctx_destroy(msb_ctx *ctx);
int msb_ctx_sync(msb_ctx *ctx);
/* Per-phase device times (ms, CUDA events on the context's stream) of the last msb_scan /
 * msb_score / msb_seqs_from_ascii on this context.  Index by MSB_T_*. */
enum { MSB_T_H2D = 0, MSB_T_ENCODE, MSB_T_PREFILTER, MSB_T_EXACT, MSB_T_ORDER, MSB_T_D2H,
       MSB_T_SCORE, MSB_T_SELECT, MSB_T_ROWS, MSB_T_ROW_SORT, MSB_T_COUNT };
int msb_ctx_timings(const msb_ctx *ctx, double *ms, int n);
/* Counters of the last msb_scan: index by MSB_C_*. */
enum { MSB_C_CANDIDATES = 0, MSB_C_DIRTY, MSB_C_HITS, MSB_C_LAUNCHES, MSB_C_RETRIES,
       MSB_C_PREFILTER_LAUNCHES, MSB_C_COUNT };
int msb_ctx_counters(const msb_ctx *ctx, int64_t *v, int n);

/* Tuning / test knobs of ONE context (nothing is process-wide): "ascii_slices" upload slices of
 * msb_scan_ascii (1..7); "tc_interleave" 0 = the prefilter's motif tiles in ascending length order instead
 * of short and long alternating (default 1); "tc_first_lane_cap" records per lane
 * buffer on the first attempt (tests of the overflow retry; 0 = sized from the input); "poison_pool" 1 =
 * recycled device buffers are filled with 0xFF (tests: nothing may rely on stale contents); "tc_prof" 1
 * = per-role cycle counters of the tensor-core prefilter on stderr; "select_pilot" 0 = msb_score_select scores
 * every sample for every motif instead of the pilot + scan scheme (A/B tests). */
int msb_ctx_set_option(msb_ctx *ctx, const char *name, int value);

/* Pinned host memory for callers that want full-speed H2D (cudaHostAlloc / cudaFreeHost). */
int msb_pinned_alloc(int64_t bytes, void **ptr);
int msb_pinned_free(void *ptr);

/* ---- motif set (replaces convert_pwm + get_max_raw_score, cscore.c:36-79) ------------------- */
/* cutoffs may be NULL: every cutoff is then 1, as in cscore.c:71-75. */
int msb_motifs_create(msb_ctx *ctx, int32_t n_motifs, const int32_t *lens, const double *mats,
                      const int64_t *mat_off, const double *cutoffs, msb_motifs **out);
int msb_motifs_set_cutoffs(msb_motifs *motifs, const double *cutoffs);
int msb_motifs_count(const msb_motifs *motifs, int32_t *n_motifs);
/* max_raw_score per motif exactly as cscore.c:36-48 computes it. */
int msb_motifs_max_raw(const msb_motifs *motifs, double *out);
int msb_motifs_destroy(msb_motifs *motifs);

/* ---- sequence set (replaces convert_seq, cscore.c:81-114) ----------------------------------- */
/* Copies the bytes to the device and encodes + packs them there. */
int msb_seqs_from_ascii(msb_ctx *ctx, int64_t n_seqs, const char *seq_bytes,
                        const int64_t *seq_off, msb_seqs **out);
/* The same from sequences that are ALREADY packed the way the library keeps them (a packed genome cache
 * on disk, another context's msb_seqs_to_packed): 0.375 B/bp cross PCIe instead of 1 B/bp, and nothing is
 * encoded.  Layout: sequence i occupies the 32-base blocks [poff_i / 32, poff_{i+1} / 32) with poff_0 = 0 and
 * poff_{i+1} = poff_i + lens[i] rounded up to 32; block b is codes[2 b], codes[2 b + 1] (2 bits per base,
 * base k of the block at bits 2 (k % 16) of word k / 16; A C G T = 0 1 2 3, cscore.c:91-108) and nmask[b]
 * (bit k set <=> base k is not A/C/G/T, cscore.c:109-110).  Bits behind a sequence's last base and codes
 * of masked bases are ignored (cleared on the device). */
#define MSB_SEQS_ASYNC 1   /* return at once: the copies run on the context's copy stream and overlap a scan in
                            * progress; `codes` / `nmask` must stay valid (and should be pinned) until the first
                            * scan of the set has returned, or msb_seqs_wait */
int msb_seqs_from_packed(msb_ctx *ctx, int64_t n_seqs, const int64_t *lens, const uint32_t *codes,
                         const uint32_t *nmask, int flags, msb_seqs **out);
int msb_seqs_wait(const msb_seqs *seqs);
/* The packed planes of a sequence set, in the layout above: 2 * B and B words, B = sum_i ceil(len_i / 32). */
int msb_seqs_to_packed(msb_ctx *ctx, const msb_seqs *seqs, uint32_t *codes, uint32_t *nmask);
/* Resident genome (SURVEY 8 f-1): instead of one host fetch per region (Scanner._extract_seq,
 * scanner.py:71-87 -> Genome.fetch_sequence -> pysam FastaFile.fetch, genome/__init__.py:135) the
 * chromosomes are encoded once into a resident msb_seqs and every later sequence set is cut out of
 * it on the device: sequence i of the result = bases [start[i], end[i]) of sequence src_idx[i] of
 * `src`, `end` clipped at the source length as fetch does (start < 0 or a bad index: MSB_EINVAL).
 * Only the 20 n bytes of the interval table cross PCIe. */
int msb_seqs_extract(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx,
                     const int64_t *start, const int64_t *end, msb_seqs **out);
/* msb_seqs_extract with bases substituted (the alternative alleles of a variant scan): after the cut, base
 * sub_pos[k] of sequence i (relative to its clipped start), k in [sub_off[i], sub_off[i + 1]), becomes the A/C/G/T
 * code sub_code[k] (0..3) and is no longer masked.  sub_off has n + 1 entries, sub_off[0] = 0; only the interval and
 * substitution tables cross PCIe. */
int msb_seqs_extract_subst(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                           const int64_t *end, const int64_t *sub_off, const int32_t *sub_pos, const uint8_t *sub_code,
                           msb_seqs **out);
/* msb_seqs_extract with a splice (the alternative alleles of a variant scan with indels): sequence i is the cut
 * interval (clipped like msb_seqs_extract) with its bases [splice_at[i], splice_at[i] + del_len[i]) replaced by the
 * A/C/G/T codes ins_code[ins_off[i] .. ins_off[i + 1]) (0..3), either side possibly empty, so it is
 * del_len[i] - (ins_off[i + 1] - ins_off[i]) bases shorter than the interval.  ins_off has n + 1 entries, ins_off[0] =
 * 0; a splice outside its interval or a code above 3 is MSB_EINVAL.  Only the tables cross PCIe. */
int msb_seqs_extract_splice(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                            const int64_t *end, const int32_t *splice_at, const int32_t *del_len, const int64_t *ins_off,
                            const uint8_t *ins_code, msb_seqs **out);
/* msb_seqs_extract with several edits per sequence (the haplotypes of a cluster of alleles): sequence i is the cut
 * interval (clipped like msb_seqs_extract) with each edit k in [edit_off[i], edit_off[i + 1]) -- its bases
 * [edit_at[k], edit_at[k] + edit_del[k]), relative to the interval -- replaced by the A/C/G/T codes
 * ins_code[ins_off[k] .. ins_off[k + 1]) (0..3).  edit_off has n + 1 entries and ins_off n_edits + 1, both starting at
 * 0.  Edits out of order, overlapping (an insertion occupies its junction: the next edit starts at or behind
 * edit_at + max(edit_del, 1)), outside their interval, or a code above 3 are MSB_EINVAL.  Only the tables cross PCIe.
 * msb_seqs_extract_splice is this call with one edit per sequence. */
int msb_seqs_extract_edits(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx, const int64_t *start,
                           const int64_t *end, const int64_t *edit_off, const int32_t *edit_at, const int32_t *edit_del,
                           const int64_t *ins_off, const uint8_t *ins_code, msb_seqs **out);
/* Number of non-ACGT bases in each of n windows [start[i], start[i] + length) of sequence src_idx[i] of a
 * resident set (clipped at the sequence end): the device half of the background sampler's acceptance
 * test `seq.count('N') + seq.count('n') <= max_n` (genome/__init__.py:172-175) -- a window without
 * any non-ACGT base is accepted without being fetched. */
int msb_seqs_window_ncount(msb_ctx *ctx, const msb_seqs *src, int64_t n, const int32_t *src_idx,
                           const int64_t *start, int32_t length, int32_t *counts);
int msb_seqs_count(const msb_seqs *seqs, int64_t *n_seqs, int64_t *total_bp);
/* True length in bases of every sequence (n_seqs entries). */
int msb_seqs_lengths(const msb_seqs *seqs, int64_t *lens);
/* Genome-wide scans cut a chromosome into chunks that overlap by (longest motif - 1) bases, so a
 * window belongs to the chunk that holds its START (the reference scans a chromosome as one
 * string, cscore.c:336-340).  limit[i] = number of leading positions of sequence i at which a
 * window may start; sites starting at or behind it are not reported.  NULL restores the default
 * (the whole sequence). */
int msb_seqs_set_start_limit(msb_seqs *seqs, const int32_t *limit);
/* Parity accessor: decode the packed device representation back to the reference's int8 codes
 * (0..3, -1) for all sequences, concatenated like the input. */
int msb_seqs_codes(msb_ctx *ctx, const msb_seqs *seqs, int8_t *codes);
int msb_seqs_destroy(msb_seqs *seqs);

/* ---- scan (replaces scan_motif_thread + scan_motif, cscore.c:317-476) ----------------------- */
/* Sites come back motif-major, then (sequence, start) ascending, forward before reverse at the
 * same start -- the order of the reference's per-motif lists.  Scores are the reference's
 * doubles bit for bit; the hit predicate is score - cutoff >= -1e-10. */
int msb_scan(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
             msb_result **out);
/* The same with flags.  MSB_SCAN_DEDUP additionally applies the reference's adjacent-site
 * de-duplication (deduplicate_motif_sites, scanner.py:156-193) on the device: per (motif,
 * sequence) and per strand, a site closer than the motif length to the previous survivor
 * replaces it only if it scores strictly higher. */
#define MSB_SCAN_DEDUP 1
/* MSB_SCAN_COUNTS: only per-motif site counts are wanted (genome-wide counting): the sites are neither
 * ordered nor kept; valid with the *_device entry points (msb_scan_device_counts reads the counts), an error
 * with the ones that return a msb_result.  Ignored together with MSB_SCAN_DEDUP (which needs the order). */
#define MSB_SCAN_COUNTS 2
/* MSB_SCAN_ASYNC: the call returns as soon as the device-to-host copy of the sites is enqueued on the
 * context's copy stream; the next scan on the same context overlaps it.  msb_result_total is valid at
 * once; msb_result_wait (or msb_result_counts / msb_result_arrays, which wait) makes the arrays valid. */
#define MSB_SCAN_ASYNC 4
/* MSB_SCAN_COMPACT: sites come back as 12 bytes (score + a uint32 holding packed position << 1 | strand bit)
 * instead of 17: a third less PCIe traffic, which is what bounds an all-sites genome-wide scan on 8 GPUs of
 * one host.  msb_result_compact hands out the raw arrays + the sequence layout that decodes them;
 * msb_result_arrays still works (the first call decodes on the host); msb_merge_sites_compact gathers such
 * results directly.  Ignored with MSB_SCAN_DEDUP and for sequence sets of 2^31 packed positions or more
 * (the result is then an ordinary one: msb_result_compact returns a NULL array). */
#define MSB_SCAN_COMPACT 8
int msb_scan_ex(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
                int flags, msb_result **out);
/* c_scan_motif in one call with persistent motifs (cscore.c:399-476: strings in, sites out):
 * msb_seqs_from_ascii + msb_scan_ex, with the host-to-device copy of the sequence bytes cut into
 * slices of whole sequences so that the copy of one slice overlaps the scan of the previous one.
 * `seq_bytes` should be pinned (msb_pinned_alloc) for the copies to be asynchronous.  The encoded
 * sequence set is returned through `seqs_out` unless that is NULL. */
int msb_scan_ascii(msb_ctx *ctx, const msb_motifs *motifs, int64_t n_seqs, const char *seq_bytes,
                   const int64_t *seq_off, int strand, int flags, msb_seqs **seqs_out, msb_result **out);
/* Range scan over a resident sequence set (genome-wide scans, configs[3]): only windows that START
 * in [start[k], end[k]) of sequence seq_idx[k] are scored; a window may run past `end` into the rest
 * of its sequence, exactly as if the whole sequence had been scanned (cscore.c:336-340), so the
 * union over a partition of a chromosome into ranges equals the unchunked scan and no overlap has
 * to be shipped.  `end` is clipped at the sequence length; ranges must not overlap (MSB_EINVAL).
 * seq_idx / start of the sites refer to `seqs`.  MSB_SCAN_DEDUP de-duplicates per range when no sequence
 * appears in more than one range of the call (MSB_EINVAL otherwise: the reference de-duplicates over a whole
 * region's site list, scanner.py:171-193, which a second range of the sequence would cut); the chains of
 * overlapping sites at the range edges are then kept for msb_scan_device_boundary_sites. */
int msb_scan_ranges(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
                    int flags, int64_t n_ranges, const int64_t *seq_idx, const int64_t *start,
                    const int64_t *end, msb_result **out);
int msb_scan_ranges_device(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
                           int flags, int64_t n_ranges, const int64_t *seq_idx, const int64_t *start,
                           const int64_t *end, int64_t *n_sites);
/* Device-only variant for measurement: same kernels, results left on the device, no D2H. */
int msb_scan_device(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
                    int flags, int64_t *n_sites);
/* Per-motif site counts of the last msb_scan_device on this context (n_motifs entries): the only
 * thing a counts-only genome-wide scan copies back. */
int msb_scan_device_counts(msb_ctx *ctx, int64_t *counts, int32_t n_motifs);
/* Per motif, the number of sequences with at least one site in the last msb_scan_device /
 * msb_scan_ranges_device on this context: the only thing motif_enrichment needs from a scan
 * (stats.py:29-31 counts the regions whose site list is non-empty), reduced on the device. */
int msb_scan_device_region_counts(msb_ctx *ctx, int64_t *counts, int32_t n_motifs);
/* Boundary chains of the last msb_scan_ranges / msb_scan_ranges_device with MSB_SCAN_DEDUP on this context
 * (MSB_EINVAL after any other scan).  A range is a piece of a longer sequence whose neighbours were scanned
 * on their own; a dedup chain (same-strand sites with consecutive starts less than the motif length L apart)
 * at a range edge may continue into a neighbour.  Per (motif, range, strand) the sites of the HEAD chain (the
 * first chain, if its first site starts less than L - 1 bases after the range start) and of the TAIL chain
 * (the last chain, if its last site starts after range end - L) come back raw, before de-duplication, in the
 * order of the scan's sites: motif, seq_idx, start (relative to the sequence), score, strand and flags
 * (bit 0: kept by the per-range de-duplication, bit 1: head chain, bit 2: tail chain; a chain that is both
 * is listed once).  *n receives the number of such sites; the arrays are filled when cap >= *n. */
int msb_scan_device_boundary_sites(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *motif, int32_t *seq_idx,
                                   int32_t *start, double *score, int8_t *strand, int8_t *flags);
/* Per (motif, sequence) cell of the last msb_scan_device / msb_scan_ranges_device on this context, reduced on
 * the device: counts[m * n_seqs + s] = number of final sites, best[...] = their best score (NaN when empty).
 * n_seqs must be the scanned set's sequence count.  Not after MSB_SCAN_COUNTS or a compact scan. */
int msb_scan_device_cell_stats(msb_ctx *ctx, int32_t n_motifs, int64_t n_seqs, int64_t *counts, double *best);
/* Variant-effect scan.  Sequence i of `ref` is allele i's context on the reference genome, sequence i of `alt` the
 * same bases with the allele substituted (msb_seqs_extract / msb_seqs_extract_subst: equal lengths); the changed
 * bases are [core_start[i], core_start[i] + core_len[i]) of it.  Both sets are scanned (msb_scan_device without
 * flags); every final site whose window overlaps its core is re-scored on the other context with the reference's
 * arithmetic and becomes a row when it is a site on at least one allele: effect 1 loss (site on ref only), 2 gain
 * (alt only), 3 both -- one row per (allele, motif, start, strand), ordered by allele, motif, start, forward before
 * reverse.  *n_rows receives the number of rows; read them with msb_scan_device_variant_rows.  Timings: prefilter /
 * exact / order summed over the two scans, MSB_T_ROWS the row kernel, MSB_T_ROW_SORT the ordering of the rows. */
int msb_scan_variants(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *ref, const msb_seqs *alt,
                      const int32_t *core_start, const int32_t *core_len, int strand, int64_t *n_rows);
/* msb_scan_variants with a core length per side (indels): the changed bases are [core_start[i], core_start[i] +
 * ref_core_len[i]) of ref context i and [core_start[i], core_start[i] + alt_core_len[i]) of alt context i (one of the two
 * may be 0, not both); the contexts must differ in length by exactly alt_core_len[i] - ref_core_len[i].  A site of length L
 * at s touches the change when s < core_start + its own side's core length and s + L > core_start (a 0-length core: the
 * window straddles the junction).  It is paired with the other context's window at s when s < core_start + the shorter
 * core length and that window fits in the other context; paired sites make rows exactly as above.  An unpaired ref site
 * is a row with effect 5 (loss, alt_score NaN), an unpaired alt site one with effect 6 (gain, ref_score NaN).  With
 * equal core lengths this is msb_scan_variants. */
int msb_scan_variants_ex(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *ref, const msb_seqs *alt,
                         const int32_t *core_start, const int32_t *ref_core_len, const int32_t *alt_core_len, int strand,
                         int64_t *n_rows);
/* msb_scan_variants_ex with several edits per context (the haplotypes of a cluster of alleles): context i carries the
 * edits k in [edit_off[i], edit_off[i + 1]) (edit_off has n + 1 entries, edit_off[0] = 0), edit k replacing the ref
 * bases [edit_at[k], edit_at[k] + edit_ref_len[k]) by edit_alt_len[k] alt bases (not both 0).  The edits of a context
 * are ordered and do not overlap (the next starts at or behind edit_at + max(edit_ref_len, 1)); on the alt context
 * edit k starts at edit_at[k] + the net length change of the edits before it.  A site of length L at s on one side is
 * affected when s < start + len and s + L > start for some edit's core on that side (a 0-length core: the window
 * straddles the junction).  Inside edit k's core at offset o < min(ref len, alt len) it maps to the other side's core
 * start + o, behind that offset it has no partner; in a stretch between cores it maps by the net shift of the edits
 * before it.  A mapped window that fits in the other context is paired.  Rows are made as by msb_scan_variants_ex and
 * ordered by context, motif, own-side start (the ref start for effect 1 / 3 / 5, the alt start for 2 / 6), strand, ref
 * before alt. */
int msb_scan_haplotypes(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *ref, const msb_seqs *alt,
                        const int64_t *edit_off, const int32_t *edit_at, const int32_t *edit_ref_len,
                        const int32_t *edit_alt_len, int strand, int64_t *n_rows);
/* The rows of the last msb_scan_variants / msb_scan_variants_ex / msb_scan_haplotypes (MSB_EINVAL after any other
 * scan): *n receives their number, the arrays are filled when cap >= *n.  start is relative to the context (for
 * msb_scan_haplotypes the own-side start); strand 1 / 2; ref_score / alt_score are the window's scores on the two
 * alleles bit for bit; effect 1 / 2 / 3 (or 5 / 6) as above.  MSB_T_D2H times the copies. */
int msb_scan_device_variant_rows(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *allele, int32_t *motif, int32_t *start,
                                 int8_t *strand, double *ref_score, double *alt_score, int8_t *effect);
/* msb_scan_device_variant_rows plus other_start: the window's start on the other side, relative to that context, or -1
 * when it has no partner there. */
int msb_scan_device_haplotype_rows(msb_ctx *ctx, int64_t cap, int64_t *n, int32_t *context, int32_t *motif, int32_t *start,
                                   int8_t *strand, double *ref_score, double *alt_score, int8_t *effect,
                                   int32_t *other_start);
int msb_result_wait(msb_result *res);
int msb_result_total(const msb_result *res, int64_t *n_sites);
int msb_result_counts(const msb_result *res, int64_t *counts /* n_motifs */);
/* Borrowed pointers into the result (valid until msb_result_destroy): n_sites entries each. */
int msb_result_arrays(const msb_result *res, const int32_t **seq_idx, const int32_t **start,
                      const double **score, const int8_t **strand /* 1 or 2 */);
/* Compact results (MSB_SCAN_COMPACT): pos_strand[i] >> 1 is the site's packed position p, sequence s owns it
 * iff poff[s] <= p < poff[s + 1] (poff: n_seqs + 1 entries, multiples of 32), start = p - poff[s];
 * pos_strand[i] & 1 = 0 forward, 1 reverse.  *pos_strand is NULL for a result that is not compact. */
int msb_result_compact(const msb_result *res, const uint32_t **pos_strand, const double **score, const int64_t **poff,
                       int64_t *n_seqs);
int msb_result_destroy(msb_result *res);

/* ---- host-side gather of several results (replaces the reference's per-motif result lists filled by
 * its thread pool, cscore.c:323-328, 425-436) ----------------------------------------------------- */
/* n_parts motif-major arrays (one per GPU or per batch, each over its own sequences, parts in ascending
 * sequence order) -> one motif-major array: for every motif, part 0's entries, then part 1's, ...
 * counts[p * n_motifs + m] = entries of motif m in part p; src[p] = part p's array of elem_size-byte entries;
 * add_i32 (optional, 4-byte entries only): per-part addend, e.g. the part's first global sequence index.
 * Pure host code (memcpy on up to n_threads threads); no device, no context. */
int msb_merge_motif_major(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const void *const *src,
                          void *dst, int32_t elem_size, const int64_t *add_i32, int32_t n_threads);
/* The same for whole site lists in one pass, with the parts' local sequence numbering translated on the way:
 * part p's sequence q (a piece of a chromosome in a sharded genome scan, a region of a block in a multi-GPU
 * region scan) becomes group seq_to_group[p][q] (its chromosome / global region) and its starts are shifted by
 * seq_offset[p][q] (the piece's first base); either table may be NULL (identity / no shift). */
int msb_merge_sites(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const int32_t *const *seq_idx,
                    const int32_t *const *start, const double *const *score, const int8_t *const *strand,
                    const int32_t *const *seq_to_group, const int32_t *const *seq_offset, int32_t *out_group,
                    int32_t *out_start, double *out_score, int8_t *out_strand, int32_t n_threads);
/* msb_merge_sites over compact results (msb_result_compact's arrays and layout per part). */
int msb_merge_sites_compact(int32_t n_parts, int32_t n_motifs, const int64_t *counts, const uint32_t *const *pos_strand,
                            const double *const *score, const int64_t *const *poff, const int64_t *n_seqs,
                            const int32_t *const *seq_to_group, const int32_t *const *seq_offset, int32_t *out_group,
                            int32_t *out_start, double *out_score, int8_t *out_strand, int32_t n_threads);

/* ---- result tables (host code; the reference builds them from nested lists, io/__init__.py:12-38) ------- */
/* Rows [r0, r1) of motif_sites_number.xls and motif_sites_score.xls as text, from a scan's motif-major arrays
 * (offsets: CSR over motifs; seq_idx ascending within a motif): row r = lead[lead_off[r - r0] .. lead_off[r - r0 + 1])
 * (the caller's "chr<TAB>start<TAB>end<TAB>") followed by one tab-separated cell per motif -- the number of sites
 * of the region, resp. the best score (`NA` without a site; doubles printed like Python's str()) -- and "\n".
 * The two buffers are malloc'ed; release them with msb_text_free.  Up to n_threads host threads. */
int msb_format_site_tables(int32_t n_motifs, const int64_t *offsets, const int32_t *seq_idx, const double *score,
                           int64_t r0, int64_t r1, const char *lead, const int64_t *lead_off, char **num_text,
                           int64_t *num_len, char **score_text, int64_t *score_len, int32_t n_threads);
/* The same rows from dense cells: counts / best are n_rows x n_motifs row-major (best ignored where the count
 * is 0); rows [0, n_rows) of lead / lead_off. */
int msb_format_cell_tables(int64_t n_rows, int32_t n_motifs, const int64_t *counts, const double *best, const char *lead,
                           const int64_t *lead_off, char **num_text, int64_t *num_len, char **score_text,
                           int64_t *score_len, int32_t n_threads);
/* One motif's motif_sites/<id>_<name>_sites.bed (io/__init__.py:41-55) written to `path`: per site, in the given
 * order, "chrom<TAB>s<TAB>s + length<TAB>.<TAB>score<TAB>strand" with chrom = names[name_off[g] .. name_off[g + 1])
 * of the site's group g, s = start + group_base[g] (group_base may be NULL), the score printed like Python's
 * str() and strand 1 -> '+', else '-'.  Formatted in blocks on up to n_threads host threads, written in order. */
int msb_write_sites_bed(const char *path, int64_t n, const int32_t *group, const int32_t *start, const int64_t *group_base,
                        const double *score, const int8_t *strand, int32_t length, int64_t n_groups, const char *names,
                        const int64_t *name_off, int32_t n_threads);
/* motif_variant_sites.xls written to `path`: `header` (may be NULL), then per row, in the given order,
 * lead[lead_off[a] .. lead_off[a + 1]) of its allele a (the caller's "chrom<TAB>pos<TAB>id<TAB>ref<TAB>alt<TAB>"),
 * motif_text[motif_off[m] .. motif_off[m + 1]) of its motif m ("id<TAB>name<TAB>"), then start, start + motif_len[m],
 * '+' / '-', ref_score, alt_score (printed like Python's str()) and loss / gain / both for effect 1 / 2 / 3,
 * tab-separated, "\n".  Effect 5 is a loss and 6 a gain whose other allele has no window (msb_scan_variants_ex): the
 * missing score is written as NA.  Any other effect is MSB_EINVAL.  Formatted in blocks on up to n_threads host threads, written in order. */
int msb_write_variant_table(const char *path, const char *header, int64_t n, const int32_t *allele, const int32_t *motif,
                            const int32_t *start, const int8_t *strand, const double *ref_score, const double *alt_score,
                            const int8_t *effect, int64_t n_alleles, const char *lead, const int64_t *lead_off, int32_t n_motifs,
                            const char *motif_text, const int64_t *motif_off, const int32_t *motif_len, int32_t n_threads);
/* motif_haplotype_sites.xls, formatted like msb_write_variant_table: per row lead[lead_off[c] .. lead_off[c + 1]) of its
 * cluster c (the caller's "chrom<TAB>cluster<TAB>ids<TAB>"), the motif text, ref_start, ref_start + motif_len[m],
 * alt_start, alt_start + motif_len[m] (NA<TAB>NA for a start below 0: no window on that side), then strand, scores and
 * effect exactly as there (effects 1 / 2 / 3 / 5 / 6, the missing score of 5 / 6 as NA). */
int msb_write_haplotype_table(const char *path, const char *header, int64_t n, const int32_t *cluster, const int32_t *motif,
                              const int64_t *ref_start, const int64_t *alt_start, const int8_t *strand, const double *ref_score,
                              const double *alt_score, const int8_t *effect, int64_t n_clusters, const char *lead,
                              const int64_t *lead_off, int32_t n_motifs, const char *motif_text, const int64_t *motif_off,
                              const int32_t *motif_len, int32_t n_threads);
int msb_text_free(char *text);

/* ---- score (replaces motif_score_thread + motif_score, cscore.c:174-302) -------------------- */
/* out is n_motifs x n_seqs row-major: the offset-0 window score of every sequence. */
int msb_score(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
              double *out);
/* Fused `motif --build` step (cli/motif.py:133-137 + motif/__init__.py:378-401): for every motif the
 * n_ranks (<= 8) order statistics sorted_descending(scores of all sequences)[ranks[k]], bit-identical to
 * sorting msb_score's rows, without ever materialising the score matrix when the ranks sit in the top
 * 1/32 of a large sample (a pilot picks per-motif thresholds, the scan path returns the samples above them
 * with their exact scores, a radix select reads the ranks).  out is n_motifs x n_ranks row-major. */
int msb_score_select(msb_ctx *ctx, const msb_motifs *motifs, const msb_seqs *seqs, int strand,
                     int32_t n_ranks, const int64_t *ranks, double *out);

/* ---- one-shot mirrors of the two reference methods ----------------------------------------- */
int msb_c_scan_motif(int device, int32_t n_motifs, const int32_t *lens, const double *mats,
                     const int64_t *mat_off, const double *cutoffs, int64_t n_seqs,
                     const char *seq_bytes, const int64_t *seq_off, int strand,
                     msb_result **out);
int msb_c_score(int device, int32_t n_motifs, const int32_t *lens, const double *mats,
                const int64_t *mat_off, int64_t n_seqs, const char *seq_bytes,
                const int64_t *seq_off, int strand, double *out);

#ifdef __cplusplus
}
#endif
#endif /* MSB200_H */
