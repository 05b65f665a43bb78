// kernels.cuh -- device code of libmsb200 (sm_100a) except the prefilter (prefilter_tc.cuh).
//
//   encode_pack_kernel      ASCII -> 2-bit codes + N mask            (cscore.c:81-114)
//   exact_records_kernel    fp64 re-score of the prefilter's candidates in the reference's
//                           accumulation order + the reference's hit predicate (cscore.c:344-389)
//   exact_dirty_kernel      the same for windows that touch a non-ACGT base
//   exact_positions_kernel  the same for motifs the prefilter cannot take (L > 64, non-finite)
//   decode_sites_kernel     sorted keys -> (seq_idx, start, strand); motif_offsets_kernel: CSR
//   dedup_flags_kernel      adjacent-site de-duplication              (scanner.py:156-193)
//   score0_kernel           offset-0 window score of every sequence     (cscore.c:191-223)
//   extract_subst_kernel    resident-genome extraction with allele bases overlaid (variant contexts)
//   extract_edits_kernel    resident-genome extraction with bases deleted and inserted (indel and haplotype contexts)
//   variant_rows_kernel     sites of the ref / alt context scans -> gain / loss / both rows
#pragma once
#include "common.cuh"

namespace msb {

// Largest s with poff[s] <= p.  Empty sequences share a start with their successor and are
// skipped because the search returns the LAST such s.
__device__ __forceinline__ int64_t find_seq(const int64_t *__restrict__ poff, int64_t n_seqs,
                                            int64_t p) {
    int64_t lo = 0, hi = n_seqs;  // invariant: poff[lo] <= p, answer in [lo, hi)
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (__ldg(poff + mid) <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// The reference's int8 code of packed position q: 0..3, or -1 for anything but ACGT/acgt.
__device__ __forceinline__ int base_code(const SeqView &S, int64_t q) {
    uint32_t m = __ldg(S.nmask + (q >> 5));
    if ((m >> (q & 31)) & 1u) return -1;
    uint32_t w = __ldg(S.codes + (q >> 4));
    return (int) ((w >> ((q & 15) * 2)) & 3u);
}

// ---------------------------------------------------------------------------------------------
// encode + pack.  One thread per 32-base block of the packed space.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
encode_pack_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ seq_off,
                   const int64_t *__restrict__ poff, const int32_t *__restrict__ len,
                   int64_t n_seqs, int64_t first_block, int64_t n_blocks, uint32_t *__restrict__ codes,
                   uint32_t *__restrict__ nmask, int32_t *__restrict__ blk_seq) {
    int64_t b = first_block + (int64_t) blockIdx.x * blockDim.x + threadIdx.x;   // blocks [first_block, n_blocks)
    if (b >= n_blocks) return;
    int64_t p = b * kPadBases;
    int64_t s = find_seq(poff, n_seqs, p);
    int64_t j = p - __ldg(poff + s);
    int n = (int) min((int64_t) kPadBases, (int64_t) __ldg(len + s) - j);
    const uint8_t *src = ascii + __ldg(seq_off + s) + j;
    uint32_t lo = 0, hi = 0, mask = 0;
#pragma unroll
    for (int k = 0; k < kPadBases; k++) {
        if (k < n) {
            uint32_t c = (uint32_t) __ldg(src + k) | 0x20u;  // fold case (cscore.c:91-108)
            uint32_t code = 0, isn = 0;
            if (c == 0x61u) code = 0;        // A a
            else if (c == 0x63u) code = 1;   // C c
            else if (c == 0x67u) code = 2;   // G g
            else if (c == 0x74u) code = 3;   // T t
            else isn = 1;                    // default: -1 (cscore.c:109-110)
            if (k < 16) lo |= code << (2 * k); else hi |= code << (2 * (k - 16));
            mask |= isn << k;
        }
    }
    codes[2 * b] = lo;
    codes[2 * b + 1] = hi;
    nmask[b] = mask;
    blk_seq[b] = (int32_t) s;
}

// ---------------------------------------------------------------------------------------------
// extract: build a packed sequence set from intervals of a resident one (the device-side
// counterpart of Scanner._extract_seq's per-region fetch, scanner.py:71-87).  One thread per
// 32-base block of the destination: 64 code bits + 32 mask bits funnel-shifted out of the source.
// ---------------------------------------------------------------------------------------------
// The bases [j, j + n) (n <= 32) of destination sequence s, cut out of the source: returns the block's two code
// words and its mask word, with every bit behind the n-th base cleared.
__device__ __forceinline__ void extract_block(const SeqView &src, const int32_t *__restrict__ src_idx,
                                              const int64_t *__restrict__ src_start, int64_t s, int64_t j, int n,
                                              uint32_t &lo, uint32_t &hi, uint32_t &mask) {
    lo = 0, hi = 0, mask = 0;
    if (n > 0) {
        const int64_t q = __ldg(src.poff + __ldg(src_idx + s)) + __ldg(src_start + s) + j;
        // the source buffers carry zero padding behind their last block (msb_seqs_from_ascii)
        const uint32_t *cp = src.codes + (q >> 4);
        const uint32_t sh = (uint32_t) (q & 15) * 2;
        const uint32_t c0 = __ldg(cp), c1 = __ldg(cp + 1), c2 = __ldg(cp + 2);
        lo = __funnelshift_r(c0, c1, sh);
        hi = __funnelshift_r(c1, c2, sh);
        const uint32_t *mp = src.nmask + (q >> 5);
        mask = __funnelshift_r(__ldg(mp), __ldg(mp + 1), (uint32_t) (q & 31));
        if (n < 32) {
            mask &= (1u << n) - 1u;
            if (n <= 16) { hi = 0; lo &= n == 16 ? 0xffffffffu : ((1u << (2 * n)) - 1u); }
            else hi &= (1u << (2 * (n - 16))) - 1u;
        }
    }
}

__global__ void __launch_bounds__(256)
extract_pack_kernel(SeqView src, const int32_t *__restrict__ src_idx, const int64_t *__restrict__ src_start,
                    const int64_t *__restrict__ poff, const int32_t *__restrict__ len, int64_t n_seqs,
                    int64_t n_blocks, uint32_t *__restrict__ codes, uint32_t *__restrict__ nmask,
                    int32_t *__restrict__ blk_seq) {
    const int64_t b = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const int64_t p = b * kPadBases;
    const int64_t s = find_seq(poff, n_seqs, p);
    const int64_t j = p - __ldg(poff + s);
    const int n = (int) min((int64_t) kPadBases, (int64_t) __ldg(len + s) - j);
    uint32_t lo, hi, mask;
    extract_block(src, src_idx, src_start, s, j, n, lo, hi, mask);
    codes[2 * b] = lo;
    codes[2 * b + 1] = hi;
    nmask[b] = mask;
    blk_seq[b] = (int32_t) s;
}

// extract with substitutions (the alternative alleles of a variant scan): the same block extraction, then the
// bases sub_pos[k] (relative to the destination sequence), k in [sub_off[s], sub_off[s + 1]), become the A/C/G/T
// codes sub_code[k] and their N bits are cleared.  A sequence carries a handful of substituted bases (an SNV or
// MNV), so every thread walks its sequence's list.
__global__ void __launch_bounds__(256)
extract_subst_kernel(SeqView src, const int32_t *__restrict__ src_idx, const int64_t *__restrict__ src_start,
                     const int64_t *__restrict__ sub_off, const int32_t *__restrict__ sub_pos,
                     const uint8_t *__restrict__ sub_code, const int64_t *__restrict__ poff,
                     const int32_t *__restrict__ len, int64_t n_seqs, int64_t n_blocks, uint32_t *__restrict__ codes,
                     uint32_t *__restrict__ nmask, int32_t *__restrict__ blk_seq) {
    const int64_t b = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const int64_t p = b * kPadBases;
    const int64_t s = find_seq(poff, n_seqs, p);
    const int64_t j = p - __ldg(poff + s);
    const int n = (int) min((int64_t) kPadBases, (int64_t) __ldg(len + s) - j);
    uint32_t lo, hi, mask;
    extract_block(src, src_idx, src_start, s, j, n, lo, hi, mask);
    for (int64_t k = __ldg(sub_off + s), k1 = __ldg(sub_off + s + 1); k < k1; k++) {
        const int64_t q = (int64_t) __ldg(sub_pos + k) - j;
        if (q < 0 || q >= n) continue;
        const uint32_t c = (uint32_t) __ldg(sub_code + k) & 3u;
        mask &= ~(1u << q);
        if (q < 16) lo = (lo & ~(3u << (2 * q))) | (c << (2 * q));
        else hi = (hi & ~(3u << (2 * (q - 16)))) | (c << (2 * (q - 16)));
    }
    codes[2 * b] = lo;
    codes[2 * b + 1] = hi;
    nmask[b] = mask;
    blk_seq[b] = (int32_t) s;
}

// extract with edits (the alternative alleles of a variant scan with indels, and the haplotypes of a cluster of
// alleles): destination sequence s is its source interval with each edit k in [edit_off[s], edit_off[s + 1]) --
// bases [at_k, at_k + del_k) of the interval, in order and not overlapping -- replaced by the A/C/G/T codes
// ins_code[ins_off[k] .. ins_off[k + 1]); edit_off == nullptr: one edit per sequence, edit s.  edit_dst[k] is where
// edit k's inserted bases start in the destination (at_k + the net length change of the edits before it).  The destination alternates flanks (source bases) and
// inserted pieces; a block finds its first piece by a binary search over its sequence's edits and walks pieces until
// it is full -- any number of them (ten adjacent SNVs put twenty pieces into one block).  A flank is cut by
// extract_block at its source offset and shifted into place; inserted bases are set directly (their mask bits stay
// clear).
__global__ void __launch_bounds__(256)
extract_edits_kernel(SeqView src, const int32_t *__restrict__ src_idx, const int64_t *__restrict__ src_start,
                     const int64_t *__restrict__ edit_off, const int32_t *__restrict__ edit_at,
                     const int32_t *__restrict__ edit_del, const int32_t *__restrict__ edit_dst,
                     const int64_t *__restrict__ ins_off, const uint8_t *__restrict__ ins_code,
                     const int64_t *__restrict__ poff, const int32_t *__restrict__ len, int64_t n_seqs,
                     int64_t n_blocks, uint32_t *__restrict__ codes, uint32_t *__restrict__ nmask,
                     int32_t *__restrict__ blk_seq) {
    const int64_t b = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const int64_t p = b * kPadBases;
    const int64_t s = find_seq(poff, n_seqs, p);
    const int64_t j = p - __ldg(poff + s);
    const int64_t dlen = __ldg(len + s), jn = j + min((int64_t) kPadBases, dlen - j);
    const int64_t e0 = edit_off ? __ldg(edit_off + s) : s, e1 = edit_off ? __ldg(edit_off + s + 1) : s + 1;
    // the first edit whose inserted piece ends behind j (these ends never decrease): the block starts in the flank
    // before it or inside its inserted piece
    int64_t lo = e0, hi = e1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(edit_dst + mid) + (__ldg(ins_off + mid + 1) - __ldg(ins_off + mid)) > j) hi = mid; else lo = mid + 1;
    }
    uint64_t code = 0;
    uint32_t mask = 0;
    int64_t d = j;
    for (int64_t k = lo; d < jn; k++) {
        // flank before edit k: destination [d, fe) = source [d - shift, ...), shift = the net change of edits < k
        const int64_t fe = k < e1 ? __ldg(edit_dst + k) : dlen;
        if (d < fe) {
            const int64_t shift = k > e0 ? __ldg(edit_dst + k - 1) + (__ldg(ins_off + k) - __ldg(ins_off + k - 1)) -
                                               (__ldg(edit_at + k - 1) + __ldg(edit_del + k - 1)) : 0;
            const int64_t d1 = min(fe, jn);
            uint32_t rl, rh, rm;
            extract_block(src, src_idx, src_start, s, d - shift, (int) (d1 - d), rl, rh, rm);
            const int q = (int) (d - j);                                 // 0 <= q < 32
            code |= ((uint64_t) rh << 32 | rl) << (2 * q);
            mask |= rm << q;
            d = d1;
        }
        if (d >= jn) break;
        // inserted bases of edit k: destination [edit_dst[k], + its length), d inside it
        const int64_t i0 = __ldg(ins_off + k), ds = __ldg(edit_dst + k);
        const int64_t d1 = min(ds + (__ldg(ins_off + k + 1) - i0), jn);
        for (; d < d1; d++) code |= (uint64_t) (__ldg(ins_code + i0 + (d - ds)) & 3u) << (2 * (d - j));
    }
    codes[2 * b] = (uint32_t) code;
    codes[2 * b + 1] = (uint32_t) (code >> 32);
    nmask[b] = mask;
    blk_seq[b] = (int32_t) s;
}

// Sequences uploaded in the packed representation (msb_seqs_from_packed) -> canonical form: bits behind a
// sequence's last base cleared in both planes, codes of non-ACGT bases cleared (N -> 0), block owners filled in.
__device__ __forceinline__ uint32_t spread_bits16(uint32_t x) {   // bit i of the low half -> bit 2 i
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}
__global__ void __launch_bounds__(256)
packed_fixup_kernel(const int64_t *__restrict__ poff, const int32_t *__restrict__ len, int64_t n_seqs,
                    int64_t n_blocks, uint32_t *__restrict__ codes, uint32_t *__restrict__ nmask,
                    int32_t *__restrict__ blk_seq) {
    const int64_t b = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const int64_t p = b * kPadBases;
    const int64_t s = find_seq(poff, n_seqs, p);
    const int64_t left = (int64_t) __ldg(len + s) - (p - __ldg(poff + s));
    const int n = left >= kPadBases ? kPadBases : (left > 0 ? (int) left : 0);
    const uint32_t valid = n >= 32 ? 0xffffffffu : ((1u << n) - 1u);
    const uint32_t mask = nmask[b] & valid;
    const uint32_t acgt = valid & ~mask;   // bases whose code counts
    codes[2 * b] &= 3u * spread_bits16(acgt & 0xffffu);
    codes[2 * b + 1] &= 3u * spread_bits16(acgt >> 16);
    nmask[b] = mask;
    blk_seq[b] = (int32_t) s;
}

// Number of non-ACGT bases in each of n windows [start, start + length) of a resident set (the
// acceptance test of the background sampler, genome/__init__.py:172-175, counts the N of a sample).
// One thread per window; the window is clipped at its sequence's end.
__global__ void __launch_bounds__(256)
window_ncount_kernel(SeqView src, const int32_t *__restrict__ src_idx, const int64_t *__restrict__ start,
                     int32_t length, int64_t n, int32_t *__restrict__ counts) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t s = __ldg(src_idx + i), a = __ldg(start + i);
    const int64_t left = (int64_t) __ldg(src.len + s) - a;
    int64_t todo = left < length ? left : length;
    int64_t q = __ldg(src.poff + s) + a;
    int32_t c = 0;
    while (todo > 0) {
        const int off = (int) (q & 31);
        const int take = (int) (todo < 32 - off ? todo : 32 - off);
        const uint32_t w = __ldg(src.nmask + (q >> 5)) >> off;
        c += __popc(take >= 32 ? w : (w & ((1u << take) - 1u)));
        q += take;
        todo -= take;
    }
    counts[i] = c;
}

// Parity accessor: packed -> int8 codes laid out like the ASCII input.
__global__ void __launch_bounds__(256)
unpack_codes_kernel(SeqView S, const int64_t *__restrict__ seq_off, int8_t *__restrict__ out) {
    int64_t p = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= S.total_packed) return;
    int64_t s = find_seq(S.poff, S.n_seqs, p);
    int64_t j = p - S.poff[s];
    if (j < S.len[s]) out[seq_off[s] + j] = (int8_t) base_code(S, p);
}

// ---------------------------------------------------------------------------------------------
// exact stage: the reference's arithmetic, verbatim (cscore.c:341-389).
// ---------------------------------------------------------------------------------------------
struct ExactParams {
    SeqView seq;
    MotifView mot;
    int strand;
    int key_shift;        // make_site_key's motif shift for this sequence set
    uint64_t *hit_key;    // motif id in the motif field
    double *hit_score;
    int64_t hit_cap;
    unsigned long long *counters;  // [2] hits
};

// Raw score of one strand of window [p, p+L): double accumulation in ascending column order,
// non-ACGT bases skipped.  No multiply on the path, so the sum is the reference's bit for bit.
__device__ __forceinline__ double exact_raw(const SeqView &S, const double *__restrict__ pw, int L,
                                            int64_t p, int rev) {
    double acc = 0.0;
    for (int c = 0; c < L; c++) {
        const int row = base_code(S, p + c);
        if (row >= 0) {
            const double v = rev ? __ldg(pw + 4 * (L - 1 - c) + (3 - row)) : __ldg(pw + 4 * c + row);
            acc = __dadd_rn(acc, v);
        }
    }
    return acc;
}

__device__ __forceinline__ void test_and_emit(const ExactParams &E, uint32_t m, int64_t p, int rev,
                                              double raw) {
    const double score = __ddiv_rn(raw, __ldg(E.mot.max_raw + m));       // cscore.c:357,374
    if (__dsub_rn(score, __ldg(E.mot.cutoff + m)) >= -1e-10) {           // cscore.c:358,375
        unsigned long long slot = atomicAdd(E.counters + 2, 1ull);
        if ((int64_t) slot < E.hit_cap) {
            E.hit_key[slot] = make_site_key(m, p, (uint32_t) rev, E.key_shift);
            E.hit_score[slot] = score;
        }
    }
}

// The bases of window [p, p + 32) as registers: 2-bit codes in a 64-bit word, N flags in 32 bits.
struct Window32 {
    uint64_t codes;
    uint32_t nmask;
};
__device__ __forceinline__ Window32 load_window32(const SeqView &S, int64_t p) {
    // the packed buffers carry >= 4 words of zero padding behind the last sequence (msb_seqs_from_ascii)
    const uint32_t *cp = S.codes + (p >> 4);
    const uint32_t sh = (uint32_t) (p & 15) * 2;
    const uint32_t c0 = __ldg(cp), c1 = __ldg(cp + 1), c2 = __ldg(cp + 2);
    Window32 w;
    w.codes = ((uint64_t) __funnelshift_r(c1, c2, sh) << 32) | __funnelshift_r(c0, c1, sh);
    const uint32_t *mp = S.nmask + (p >> 5);
    w.nmask = __funnelshift_r(__ldg(mp), __ldg(mp + 1), (uint32_t) (p & 31));
    return w;
}
// exact_raw over a register window (L <= 32): same additions in the same order.
__device__ __forceinline__ double exact_raw_w(const Window32 &w, const double *__restrict__ pw, int L, int rev) {
    double acc = 0.0;
    for (int c = 0; c < L; c++) {
        if ((w.nmask >> c) & 1u) continue;
        const int row = (int) ((w.codes >> (2 * c)) & 3u);
        const double v = rev ? __ldg(pw + 4 * (L - 1 - c) + (3 - row)) : __ldg(pw + 4 * c + row);
        acc = __dadd_rn(acc, v);
    }
    return acc;
}

// The tensor-core prefilter leaves its candidate records in one buffer per epilogue lane
// (prefilter_tc.cuh, "Candidate emission").  lane_totals_kernel: counters[0] += records held (counts
// clamped to the buffer capacity), counters[3] = max(largest unclamped count) -- beyond the capacity
// the host repeats the prefilter with larger buffers.  Both counters are zero before the launch.
__global__ void __launch_bounds__(1024)
lane_totals_kernel(const uint32_t *__restrict__ lane_count, int32_t n_lanes, int64_t cap,
                   unsigned long long *__restrict__ counters) {
    __shared__ unsigned long long s_sum[32];
    __shared__ unsigned int s_max[32];
    unsigned long long sum = 0;
    unsigned int mx = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_lanes; i += gridDim.x * blockDim.x) {
        const unsigned int c = __ldg(lane_count + i);
        mx = max(mx, c);
        sum += min((unsigned long long) c, (unsigned long long) cap);
    }
    for (int d = 16; d; d >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, d);
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    }
    if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_max[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x < 32) {
        sum = s_sum[threadIdx.x];
        mx = s_max[threadIdx.x];
        for (int d = 16; d; d >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, d);
            mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        }
        if (threadIdx.x == 0) {
            atomicAdd(counters + 0, sum);
            atomicMax(counters + 3, (unsigned long long) mx);
        }
    }
}

// One warp per lane buffer, one thread per record = one window: its bases are loaded once and every
// flagged column of the chunk's 64 is decoded (col_info: tile column -> sorted motif, strand) and
// re-scored.  A warp's 32 records are contiguous (512 B).
__device__ __forceinline__ void exact_record(const ExactParams &E, const uint4 r, const int32_t *__restrict__ order,
                                             const uint32_t *__restrict__ col_info) {
    const int64_t p = (int64_t) (((uint64_t) (r.y & 0x1ffu) << 32) | r.x);
    const uint32_t col0 = r.y >> 9;
    const int64_t s = __ldg(E.seq.blk_seq + (p >> 5));
    const int64_t j = p - __ldg(E.seq.poff + s);
    const int64_t slen = __ldg(E.seq.len + s);
    if (E.seq.limit && j >= (int64_t) __ldg(E.seq.limit + s)) return;   // the next chunk owns this start
    const Window32 w = load_window32(E.seq, p);
    unsigned long long bits = ((unsigned long long) r.w << 32) | r.z;   // one flat loop: less divergence than word by word
    while (bits) {
        const int i = __ffsll((long long) bits) - 1;   // bit 32 h + 8 q + k <=> column 32 h + 4 k + q
        bits &= bits - 1;
        const uint32_t info = __ldg(col_info + col0 + (i & 32) + 4 * (i & 7) + ((i >> 3) & 3));
        if (info == 0xffffffffu) continue;   // padding column of a tile
        const uint32_t m = (uint32_t) __ldg(order + (info >> 1));
        const int rev = (int) (info & 1u);
        const int L = __ldg(E.mot.len + m);
        if (j + L > slen) continue;   // cscore.c:340
        const double *pw = E.mot.pwm + 4 * (int64_t) __ldg(E.mot.col_off + m);
        // the register window holds 32 bases; a longer motif (prefiltered on its first 32 columns) reads memory
        test_and_emit(E, m, p, rev, L <= kMaxFastLen ? exact_raw_w(w, pw, L, rev) : exact_raw(E.seq, pw, L, p, rev));
    }
}

__global__ void __launch_bounds__(256)
exact_records_kernel(ExactParams E, const uint4 *__restrict__ rec, int64_t rec_cap,
                     const uint32_t *__restrict__ lane_count, int32_t n_lanes,
                     const int32_t *__restrict__ order, const uint32_t *__restrict__ col_info) {
    const int64_t b = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= n_lanes) return;
    const int64_t n = min((int64_t) __ldg(lane_count + b), rec_cap);
    const uint4 *buf = rec + b * rec_cap;
    for (int64_t k = threadIdx.x & 31; k < n; k += 32) exact_record(E, __ldg(buf + k), order, col_info);
}

// One thread per (listed position, motif); consecutive threads take consecutive motifs of the
// same position.  `motif_ids` == nullptr means all motifs.
__global__ void __launch_bounds__(256)
exact_positions_kernel(ExactParams E, const int64_t *__restrict__ pos, int64_t n_pos, int64_t pos_base,
                       const int32_t *__restrict__ motif_ids, int32_t n_ids) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t d = t / n_ids;
    if (d >= n_pos) return;
    const uint32_t m = motif_ids ? (uint32_t) __ldg(motif_ids + (t - d * n_ids)) : (uint32_t) (t - d * n_ids);
    const int64_t p = pos ? __ldg(pos + d) : pos_base + d;
    if (p >= E.seq.total_packed) return;
    const int64_t s = find_seq(E.seq.poff, E.seq.n_seqs, p);
    const int64_t j = p - __ldg(E.seq.poff + s);
    const int L = __ldg(E.mot.len + m);
    const int64_t slen = __ldg(E.seq.len + s);
    if (j >= slen || j + L > slen) return;   // cscore.c:337,340
    if (E.seq.limit && j >= (int64_t) __ldg(E.seq.limit + s)) return;
    const double *pw = E.mot.pwm + 4 * (int64_t) __ldg(E.mot.col_off + m);
    if (E.strand & 1) test_and_emit(E, m, p, 0, exact_raw(E.seq, pw, L, p, 0));
    if (E.strand & 2) test_and_emit(E, m, p, 1, exact_raw(E.seq, pw, L, p, 1));
}

// Dirty windows (they touch a non-ACGT base) x the prefilter-path motifs.  A block takes a chunk of
// kDirtyMotifs motifs, whose fp32 matrices it stages in shared memory, and 8 x 32 listed positions:
// one position per lane (the window's bases in registers), each warp walking the chunk's motifs
// together, so the motif, its length and the column are warp-uniform and the 32 lanes' reads of one
// column hit at most 4 words of one 16-byte line.  (Reading the matrices straight from global memory
// left one sector in flight per warp: 0.71 ms for 26.6 k positions x 750 motifs; staged: see
// profiles/.)  Windows are screened in fp32 (upload_floors in msb200.cu); the few that can reach the
// cutoff are re-scored with the reference's fp64 arithmetic from global memory.
constexpr int kDirtyMotifs = 64;
constexpr int kDirtyStride = 4 * kMaxFastLen;   // floats per staged motif
__global__ void __launch_bounds__(256)
exact_dirty_kernel(ExactParams E, const int64_t *__restrict__ pos, int64_t n_pos,
                   const int32_t *__restrict__ motif_ids, int32_t n_ids) {
    __shared__ float s_pw[kDirtyMotifs * kDirtyStride];
    __shared__ float s_floor[kDirtyMotifs];
    __shared__ int32_t s_len[kDirtyMotifs];
    __shared__ uint32_t s_motif[kDirtyMotifs];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int32_t n_chunks = (n_ids + kDirtyMotifs - 1) / kDirtyMotifs;
    const int32_t chunk = (int32_t) (blockIdx.x % (unsigned) n_chunks);
    const int64_t group = (int64_t) (blockIdx.x / (unsigned) n_chunks) * 8 + wib;
    const int32_t k0 = chunk * kDirtyMotifs, n_here = min(n_ids - k0, kDirtyMotifs);
    for (int32_t kl = wib; kl < n_here; kl += 8) {
        const uint32_t m = (uint32_t) __ldg(motif_ids + k0 + kl);
        const int L = __ldg(E.mot.len + m);
        const float *src = E.mot.pwm32 + 4 * (int64_t) __ldg(E.mot.col_off + m);
        if (L <= kMaxFastLen)   // longer motifs are not screened: they go straight to the fp64 path below
            for (int i = lane; i < 4 * L; i += 32) s_pw[kl * kDirtyStride + i] = __ldg(src + i);
        if (lane == 0) { s_len[kl] = L; s_floor[kl] = __ldg(E.mot.floor32 + m); s_motif[kl] = m; }
    }
    __syncthreads();
    if (group * 32 >= n_pos) return;
    const int64_t d = group * 32 + lane;
    int64_t p = 0, left = 0;
    Window32 w;
    w.codes = 0;
    w.nmask = 0;
    if (d < n_pos) {
        p = __ldg(pos + d);
        const int64_t s = __ldg(E.seq.blk_seq + (p >> 5));
        const int64_t j = p - __ldg(E.seq.poff + s);
        left = (int64_t) __ldg(E.seq.len + s) - j;
        if (E.seq.limit && j >= (int64_t) __ldg(E.seq.limit + s)) left = 0;   // the next chunk owns this start
        if (left > 0) w = load_window32(E.seq, p);
    }
    for (int32_t kl = 0; kl < n_here; kl++) {
        const int L = s_len[kl];
        if (L > kMaxFastLen) {   // warp-uniform: a long motif, scored from memory with the reference's arithmetic
            if (L <= left) {
                const uint32_t m = s_motif[kl];
                const double *pw = E.mot.pwm + 4 * (int64_t) __ldg(E.mot.col_off + m);
                if (E.strand & 1) test_and_emit(E, m, p, 0, exact_raw(E.seq, pw, L, p, 0));
                if (E.strand & 2) test_and_emit(E, m, p, 1, exact_raw(E.seq, pw, L, p, 1));
            }
            continue;
        }
        const float *pw32 = s_pw + kl * kDirtyStride;
        // fp32 screen of both strands (FP64 issues at a fraction of the FP32 rate and the division in
        // test_and_emit is a subroutine): a score below the floor cannot pass
        // Unrolled over the columns with compile-time shifts and offsets: per column and lane one bit
        // field extract, two address adds, two shared loads and two predicated adds (the kernel is
        // issue-bound: 7e8 column steps per scan of configs[1]).
        float f32 = 0.f, r32 = 0.f;
        const float *rev_end = pw32 + 4 * (L - 1) + 3;   // reverse strand reads matrix column L - 1 - c, row 3 - row
        const uint32_t lo = (uint32_t) w.codes, hi = (uint32_t) (w.codes >> 32);
#pragma unroll
        for (int c = 0; c < kMaxFastLen; c++) {
            if (c >= L) break;   // warp-uniform
            const uint32_t row = ((c < 16 ? lo : hi) >> (2 * (c & 15))) & 3u;
            const float vf = pw32[4 * c + row], vr = *(rev_end - 4 * c - row);
            if (!((w.nmask >> c) & 1u)) { f32 += vf; r32 += vr; }
        }
        if (L > left) continue;   // cscore.c:337,340 (also lanes without a position: left = 0)
        const float floor32 = s_floor[kl];
        const bool try_f = (E.strand & 1) && !(f32 < floor32), try_r = (E.strand & 2) && !(r32 < floor32);
        if (try_f || try_r) {   // rare: the reference's arithmetic, matrices from global memory
            const uint32_t m = s_motif[kl];
            const double *pw = E.mot.pwm + 4 * (int64_t) __ldg(E.mot.col_off + m);
            if (try_f) test_and_emit(E, m, p, 0, exact_raw_w(w, pw, L, 0));
            if (try_r) test_and_emit(E, m, p, 1, exact_raw_w(w, pw, L, 1));
        }
    }
}

__global__ void __launch_bounds__(256)
decode_sites_kernel(SeqView S, const uint64_t *__restrict__ key, int64_t n, int key_shift,
                    int32_t *__restrict__ seq_idx, int32_t *__restrict__ start,
                    int8_t *__restrict__ strand) {
    int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = key[i];
    const int64_t p = site_pos(k, key_shift);
    const int64_t s = __ldg(S.blk_seq + (p >> 5));   // a site's position lies inside a sequence, so its block has an owner
    seq_idx[i] = (int32_t) s;
    start[i] = (int32_t) (p - __ldg(S.poff + s));
    strand[i] = (int8_t) (key_rev(k) + 1);  // 1 forward, 2 reverse (cscore.c:359,376)
}

// MSB_SCAN_COMPACT: a site's packed position and strand are the low key_shift (<= 32) bits of its sorted key
// (make_site_key); 4 bytes per site cross PCIe instead of 9 and the host finds the owning sequence.
__global__ void __launch_bounds__(256)
compact_sites_kernel(const uint64_t *__restrict__ key, int64_t n, int key_shift, uint32_t *__restrict__ out) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint32_t) (key[i] & ((1ull << key_shift) - 1ull));
}

// offsets[m] = first sorted site whose motif id is >= m  (m = 0..n_motifs): CSR over motifs.
__global__ void __launch_bounds__(256)
motif_offsets_kernel(const uint64_t *__restrict__ key, int64_t n, int32_t n_motifs, int key_shift,
                     int64_t *__restrict__ offsets) {
    const int32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m > n_motifs) return;
    int64_t lo = 0, hi = n;  // first i with site_motif(key[i]) >= m
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t) site_motif(__ldg(key + mid), key_shift) < (int64_t) m) lo = mid + 1; else hi = mid;
    }
    offsets[m] = lo;
}

// MSB_SCAN_COUNTS: per-motif site counts straight from the unsorted hit keys (a block-private histogram in
// shared memory when the motif set fits, flushed with one global atomic per non-empty bin).
__global__ void __launch_bounds__(256)
count_hits_kernel(const uint64_t *__restrict__ key, int64_t n, int key_shift, int32_t n_motifs, int in_smem,
                  unsigned long long *__restrict__ counts) {
    extern __shared__ unsigned int s_hist[];
    if (in_smem) {
        for (int32_t m = threadIdx.x; m < n_motifs; m += blockDim.x) s_hist[m] = 0;
        __syncthreads();
    }
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t m = site_motif(__ldg(key + i), key_shift);
        if (in_smem) atomicAdd(s_hist + m, 1u); else atomicAdd(counts + m, 1ull);
    }
    if (in_smem) {
        __syncthreads();
        for (int32_t m = threadIdx.x; m < n_motifs; m += blockDim.x)
            if (s_hist[m]) atomicAdd(counts + m, (unsigned long long) s_hist[m]);
    }
}

// Per motif, the number of sequences with at least one site (what motif_enrichment counts,
// stats.py:29-31), from the sorted site list: a site opens a new (motif, sequence) cell if it is the
// first of its motif or its sequence differs from the previous site's.
__global__ void __launch_bounds__(256)
region_counts_kernel(const uint64_t *__restrict__ key, const int32_t *__restrict__ seq_idx, int64_t n,
                     int key_shift, unsigned long long *__restrict__ out) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t m = site_motif(key[i], key_shift);
    if (i == 0 || site_motif(key[i - 1], key_shift) != m || seq_idx[i - 1] != seq_idx[i]) atomicAdd(out + m, 1ull);
}

// ---------------------------------------------------------------------------------------------
// De-duplication of adjacent sites (scanner.py:156-193), on the sorted site list.
// Per (motif, sequence) segment and per strand separately, walking sites by ascending start with
// one "current survivor": a site closer than the motif length to the survivor replaces it only
// if its score is strictly higher (`curr.score >= next.score` keeps curr, scanner.py:163).
// The surviving forward and reverse sites keep their (start, forward-first) order, which is the
// reference's `fwd + rev` followed by a stable sort on start (scanner.py:190-191).
//
// The walk only carries state across same-strand sites that are closer than the motif length to their
// predecessor (the survivor is never behind the predecessor's predecessor chain), so a segment falls
// apart into independent CHAINS at every same-strand gap >= L.  One thread per site: it looks back (at most
// the few sites within L positions) to see whether it opens a chain, and if so walks that chain.  Whole
// chromosomes de-duplicate as fast as 1 kb regions; only a run of overlapping sites is sequential.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
dedup_flags_kernel(const uint64_t *__restrict__ key, const int32_t *__restrict__ seq_idx,
                   const int32_t *__restrict__ start, const int8_t *__restrict__ strand,
                   const double *__restrict__ score, int64_t n, const int32_t *__restrict__ mlen, int key_shift,
                   int32_t *__restrict__ keep) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t m = site_motif(key[i], key_shift);
    const int32_t s = seq_idx[i];
    const int32_t L = __ldg(mlen + m);
    const int8_t which = strand[i];
    for (int64_t t = i - 1; t >= 0; t--) {   // does a same-strand site of this segment sit less than L before this one?
        if (site_motif(key[t], key_shift) != m || seq_idx[t] != s) break;
        if (start[i] - start[t] >= L) break;
        if (strand[t] == which) return;      // not a chain head: the head's thread reaches this site
    }
    int64_t cur = i, last = i;
    keep[i] = 1;
    for (int64_t t = i + 1; t < n; t++) {
        if (site_motif(key[t], key_shift) != m || seq_idx[t] != s) break;
        if (strand[t] != which) continue;
        if (start[t] - start[last] >= L) break;   // the next chain
        last = t;
        if (start[t] - start[cur] < L) {
            if (score[cur] >= score[t]) { keep[t] = 0; continue; }
            keep[cur] = 0;
        }
        keep[t] = 1;
        cur = t;
    }
}

__global__ void __launch_bounds__(256)
scatter_kept_kernel(const int32_t *__restrict__ keep, const int64_t *__restrict__ dst, int64_t n,
                    const uint64_t *__restrict__ key, const double *__restrict__ score,
                    const int32_t *__restrict__ seq_idx, const int32_t *__restrict__ start,
                    const int8_t *__restrict__ strand, uint64_t *__restrict__ o_key,
                    double *__restrict__ o_score, int32_t *__restrict__ o_seq,
                    int32_t *__restrict__ o_start, int8_t *__restrict__ o_strand) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !keep[i]) return;
    const int64_t j = dst[i];
    o_key[j] = key[i];
    o_score[j] = score[i];
    o_seq[j] = seq_idx[i];
    o_start[j] = start[i];
    o_strand[j] = strand[i];
}

// ---------------------------------------------------------------------------------------------
// c_score: offset-0 window of every sequence (cscore.c:191-223).  One thread per sequence,
// looping over a slice of motifs; out[m * n_seqs + i].
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
score0_kernel(SeqView S, MotifView M, int strand, int32_t m_begin, int32_t m_end, int64_t out_stride,
              double *__restrict__ out) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S.n_seqs) return;
    const int64_t p = __ldg(S.poff + i);
    for (int32_t m = m_begin + (int32_t) blockIdx.y; m < m_end; m += (int32_t) gridDim.y) {
        const int L = __ldg(M.len + m);
        const double *pw = M.pwm + 4 * (int64_t) __ldg(M.col_off + m);
        double f = 0.0, r = 0.0;
        for (int c = 0; c < L; c++) {
            const int row = base_code(S, p + c);
            if (row >= 0) {
                if (strand & 1) f = __dadd_rn(f, __ldg(pw + 4 * c + row));
                if (strand & 2) r = __dadd_rn(r, __ldg(pw + 4 * (L - 1 - c) + (3 - row)));
            }
        }
        double sc = 0.0;
        if (strand == 1) sc = f;
        else if (strand == 2) sc = r;
        else if (strand == 3) sc = (f > r) ? f : r;  // cscore.c:215-221
        out[(int64_t) (m - m_begin) * out_stride + i] = __ddiv_rn(sc, __ldg(M.max_raw + m));
    }
}

// ---------------------------------------------------------------------------------------------
// Order statistics of score distributions (get_score_cutoffs, motif/__init__.py:378-401: sort
// descending, read a handful of indices) by radix SELECT instead of a sort.
//
// order_key: the bijection double -> uint64 whose unsigned order is the order a radix sort of doubles
// uses (negative values below positive ones, -0.0 below +0.0, NaNs at the ends by bit pattern), so the
// selected values are the ones msb_score_select's former cub::DeviceSegmentedRadixSort returned.
// Key 0 (the bit pattern of a negative NaN with every payload bit set) marks a dead entry.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t order_key(double v) {
    const uint64_t b = (uint64_t) __double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double order_key_inv(uint64_t k) {
    const uint64_t b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long) b);
}

constexpr int kSelMaxRanks = 8;
constexpr int kSelThreads = 512;

// One block per segment.  Segment s holds the keys (kFromDoubles: doubles, keyed on the fly) at
// data[begin .. end) with begin = seg_off ? seg_off[s] : s * stride and end = seg_off ? seg_off[s + 1] :
// begin + stride.  out[s * n_ranks + j] = the ranks[j]-th largest value (0-based), found digit by digit
// from the top: per 8-bit digit one pass over the segment builds, for every group of ranks that still share
// a prefix, the histogram of the next digit among the keys with that prefix; the bucket that holds the rank
// extends the prefix.  Eight passes for all ranks together; the segment is staged in shared memory when
// it fits (smem_keys), else re-read from L2.  Warp-level vote merges equal digits before the
// shared-memory atomic: score keys share their top bytes.  ok[s] (optional) = 0 when some rank is not
// below live[s] (the number of entries that are not dead).
template <bool kFromDoubles>
__global__ void __launch_bounds__(kSelThreads)
select_ranks_kernel(const void *__restrict__ data, const int64_t *__restrict__ seg_off, int64_t stride,
                    const int64_t *__restrict__ ranks, int n_ranks, int smem_keys, const int64_t *__restrict__ live,
                    double *__restrict__ out, int32_t *__restrict__ ok) {
    extern __shared__ __align__(16) uint64_t s_keys[];
    __shared__ unsigned int s_hist[kSelMaxRanks][256];
    __shared__ uint64_t s_prefix[kSelMaxRanks];
    __shared__ long long s_rank[kSelMaxRanks];
    __shared__ int s_group[kSelMaxRanks], s_ngroups;
    const int seg = blockIdx.x;
    const int64_t begin = seg_off ? seg_off[seg] : (int64_t) seg * stride;
    const int64_t n = seg_off ? seg_off[seg + 1] - begin : stride;
    const int64_t n_live = live ? live[seg] : n;
    const uint64_t *keys = reinterpret_cast<const uint64_t *>(data) + begin;
    const double *vals = reinterpret_cast<const double *>(data) + begin;
    const bool staged = n <= (int64_t) smem_keys;
    if (staged)
        for (int64_t i = threadIdx.x; i < n; i += kSelThreads) s_keys[i] = kFromDoubles ? order_key(vals[i]) : keys[i];
    if (threadIdx.x < n_ranks) {
        s_prefix[threadIdx.x] = 0;
        s_rank[threadIdx.x] = ranks[threadIdx.x];
    }
    if (threadIdx.x == 0) {
        bool fine = true;
        for (int j = 0; j < n_ranks; j++) fine = fine && ranks[j] >= 0 && ranks[j] < n_live;
        if (ok) ok[seg] = fine ? 1 : 0;
        s_ngroups = fine ? 1 : 0;
        for (int j = 0; j < n_ranks; j++) s_group[j] = 0;
    }
    __syncthreads();
    if (s_ngroups == 0) {   // not enough live entries: the caller takes another path for this segment
        if (threadIdx.x < n_ranks) out[(int64_t) seg * n_ranks + threadIdx.x] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    for (int shift = 56; shift >= 0; shift -= 8) {
        const int ng = s_ngroups;
        for (int i = threadIdx.x; i < ng * 256; i += kSelThreads) (&s_hist[0][0])[i] = 0;
        __syncthreads();
        const uint64_t mask = shift == 56 ? 0ull : (~0ull << (shift + 8));
        // group g's prefix = the prefix of its first rank
        uint64_t gp[kSelMaxRanks];
        {
            int g = 0;
            for (int j = 0; j < n_ranks && g < ng; j++)
                if (s_group[j] == g) gp[g++] = s_prefix[j];
        }
        const int64_t n_round = (n + 31) / 32 * 32;   // whole warps take part in the vote
        for (int64_t i = threadIdx.x; i < n_round; i += kSelThreads) {
            const bool have = i < n;
            const uint64_t k = !have ? 0ull : (staged ? s_keys[i] : (kFromDoubles ? order_key(vals[i]) : keys[i]));
            int g = -1;
            if (have)
                for (int t = 0; t < ng; t++)
                    if ((k & mask) == gp[t]) g = t;
            // lanes with the same (group, digit) elect one to add their number
            const unsigned int tag = g < 0 ? 0xffffffffu : (unsigned int) (g * 256 + (int) ((k >> shift) & 255));
            const unsigned int peers = __match_any_sync(0xffffffffu, tag);
            if (g >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[0][0] + tag, (unsigned int) __popc(peers));
        }
        __syncthreads();
        if (threadIdx.x < n_ranks) {
            const int j = threadIdx.x;
            const unsigned int *h = s_hist[s_group[j]];
            long long r = s_rank[j], above = 0;
            int b = 255;
            for (; b > 0; b--) {
                if (above + (long long) h[b] > r) break;
                above += h[b];
            }
            s_rank[j] = r - above;
            s_prefix[j] |= (uint64_t) b << shift;
        }
        __syncthreads();
        if (threadIdx.x == 0) {   // regroup: ranks with equal prefixes share a histogram in the next pass
            int ngn = 0;
            for (int j = 0; j < n_ranks; j++) {
                int g = -1;
                for (int t = 0; t < j; t++)
                    if (s_prefix[t] == s_prefix[j]) { g = s_group[t]; break; }
                s_group[j] = g >= 0 ? g : ngn++;
            }
            s_ngroups = ngn;
        }
        __syncthreads();
    }
    if (threadIdx.x < n_ranks) out[(int64_t) seg * n_ranks + threadIdx.x] = order_key_inv(s_prefix[threadIdx.x]);
}

// After a scan with a start limit of 1 (only the offset-0 window of every sample) the sorted site list holds,
// per motif, one site per (sample, strand) that reached the pilot cutoff.  c_score's value for strand 3 is the
// better strand (cscore.c:215-221): key[i] = order_key(max over the sample's sites); the second site of a
// sample becomes a dead entry (key 0) and is counted in dead[motif].
__global__ void __launch_bounds__(256)
sample_keys_kernel(const uint64_t *__restrict__ site_key, const int32_t *__restrict__ seq_idx,
                   const double *__restrict__ score, int64_t n, int key_shift, uint64_t *__restrict__ key,
                   unsigned long long *__restrict__ dead) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t m = site_motif(site_key[i], key_shift);
    const int32_t s = seq_idx[i];
    if (i > 0 && site_motif(site_key[i - 1], key_shift) == m && seq_idx[i - 1] == s) {
        key[i] = 0;
        atomicAdd(dead + m, 1ull);
        return;
    }
    uint64_t k = order_key(score[i]);
    if (i + 1 < n && site_motif(site_key[i + 1], key_shift) == m && seq_idx[i + 1] == s) k = max(k, order_key(score[i + 1]));
    key[i] = k;
}

// live[m] = offsets[m + 1] - offsets[m] - dead[m]
__global__ void __launch_bounds__(256)
live_counts_kernel(const int64_t *__restrict__ offsets, const unsigned long long *__restrict__ dead, int32_t n_motifs,
                   int64_t *__restrict__ live) {
    const int32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < n_motifs) live[m] = offsets[m + 1] - offsets[m] - (int64_t) dead[m];
}

// fill an int32 array with one value (the start limit of the offset-0 scan)
__global__ void __launch_bounds__(256) fill_i32_kernel(int32_t *__restrict__ p, int64_t n, int32_t v) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// Boundary chains of a de-duplicated range scan.  A range [lo, hi) (packed positions) is a piece of a
// longer sequence; the dedup chains of its edges may continue into the neighbouring pieces, which were
// resolved on their own.  Per (motif, range) cell and strand, the HEAD chain (the first chain, when its
// first site starts less than L - 1 bases into the range: a site of the preceding piece may sit less than
// L before it) and the TAIL chain (the last chain, when its last site starts after hi - L) are emitted raw,
// with their keep flags, so that the host can re-run the greedy rule over the joined chain.
// One thread per cell; the walks never go further than the chains plus L positions.
// Emitted flag bits: 1 kept by the device, 2 in the head chain, 4 in the tail chain.
// mode 0: count[cell] = sites to emit; mode 1: write them at dst[cell] in site order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
boundary_chains_kernel(const uint64_t *__restrict__ key, const int32_t *__restrict__ seq_idx,
                       const int32_t *__restrict__ start, const int8_t *__restrict__ strand,
                       const double *__restrict__ score, const int32_t *__restrict__ keep, int64_t n,
                       const int64_t *__restrict__ r_lo, const int64_t *__restrict__ r_hi, int64_t n_ranges,
                       int32_t n_motifs, const int32_t *__restrict__ mlen, int key_shift, int mode,
                       int64_t *__restrict__ count, const int64_t *__restrict__ dst, int32_t *__restrict__ o_motif,
                       int32_t *__restrict__ o_seq, int32_t *__restrict__ o_start, double *__restrict__ o_score,
                       int8_t *__restrict__ o_strand, int8_t *__restrict__ o_flags) {
    const int64_t cell = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= (int64_t) n_motifs * n_ranges) return;
    const uint32_t m = (uint32_t) (cell / n_ranges);
    const int64_t r = cell % n_ranges, lo_p = r_lo[r], hi_p = r_hi[r];
    const int32_t L = __ldg(mlen + m);
    auto lower = [&](uint64_t k) {
        int64_t a = 0, b = n;
        while (a < b) { const int64_t mid = (a + b) >> 1; if (key[mid] < k) a = mid + 1; else b = mid; }
        return a;
    };
    const int64_t a = lower(make_site_key(m, lo_p, 0, key_shift)), b = lower(make_site_key(m, hi_p, 0, key_shift));
    int64_t emitted = 0;
    if (b <= a) { if (mode == 0) count[cell] = 0; return; }
    // head_end[x]: index of the last site of strand x's head chain (-1: none); tail_begin[x]: first site of its tail chain (n: none)
    int64_t head_end[2] = {-1, -1}, tail_begin[2] = {n, n};
    for (int x = 0; x < 2; x++) {
        int64_t last = -1;
        for (int64_t t = a; t < b; t++) {   // position tests first: they also end the walk on the other strand's sites
            const int64_t p = site_pos(key[t], key_shift);
            if (last < 0 ? p - lo_p >= L - 1 : p - site_pos(key[last], key_shift) >= L) break;
            if ((int) key_rev(key[t]) == x) last = t;
        }
        head_end[x] = last;
        int64_t first = n;
        for (int64_t t = b - 1; t >= a; t--) {
            const int64_t p = site_pos(key[t], key_shift);
            if (first == n ? p <= hi_p - L : site_pos(key[first], key_shift) - p >= L) break;
            if ((int) key_rev(key[t]) == x) first = t;
        }
        tail_begin[x] = first;
    }
    const int64_t h1 = max(head_end[0], head_end[1]);
    const int64_t t0 = min(tail_begin[0], tail_begin[1]);
    int64_t at = mode ? dst[cell] : 0;
    for (int64_t t = a; t < b; t++) {
        if (t > h1 && t < t0) { t = t0 - 1; continue; }   // the middle of the cell: nothing there to emit
        const int x = (int) key_rev(key[t]);
        const int fl = (t <= head_end[x] ? 2 : 0) | (t >= tail_begin[x] ? 4 : 0);
        if (!fl) continue;
        if (mode) {
            o_motif[at] = (int32_t) m;
            o_seq[at] = seq_idx[t];
            o_start[at] = start[t];
            o_score[at] = score[t];
            o_strand[at] = strand[t];
            o_flags[at] = (int8_t) (fl | (keep[t] ? 1 : 0));
            at++;
        }
        emitted++;
    }
    if (mode == 0) count[cell] = emitted;
}

// Per (motif, sequence) cell of a scan's final (motif, sequence)-ordered sites: the number of sites and the best
// score as an order_key (signed scores compare correctly as unsigned keys).  One thread per run of 32 sites, which
// sums runs of one cell locally: the sites are sorted, so the atomics are one per cell boundary, not per site.
__global__ void __launch_bounds__(256)
cell_stats_kernel(const uint64_t *__restrict__ key, const int32_t *__restrict__ seq_idx, const double *__restrict__ score,
                  int64_t n, int key_shift, int64_t n_seqs, unsigned long long *__restrict__ count,
                  unsigned long long *__restrict__ best) {
    const int64_t i0 = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) * 32;
    if (i0 >= n) return;
    const int64_t i1 = min(i0 + 32, n);
    int64_t cell = -1;
    unsigned long long c = 0, k = 0;
    for (int64_t i = i0; i < i1; i++) {
        const int64_t ci = (int64_t) site_motif(key[i], key_shift) * n_seqs + seq_idx[i];
        if (ci != cell) {
            if (cell >= 0) { atomicAdd(count + cell, c); atomicMax(best + cell, k); }
            cell = ci, c = 0, k = 0;
        }
        c++;
        k = max(k, (unsigned long long) order_key(score[i]));
    }
    atomicAdd(count + cell, c);
    atomicMax(best + cell, k);
}

// ---------------------------------------------------------------------------------------------
// Variant rows (msb_scan_variants_ex, msb_scan_haplotypes).  Sequence i of `ref` and of `alt` is context i on the
// reference and with its edits applied; both start at the same base.  Edit k in [edit_off[i], edit_off[i + 1])
// replaces the ref bases [R.at[k], R.at[k] + R.len[k]) by the alt bases [A.at[k], A.at[k] + A.len[k]); A.at is R.at
// shifted by the net length change of the edits before k (edit_off == nullptr: one edit per context, edit i, and
// A.at == R.at).  The edits are ordered and do not overlap, so on each side
// both their starts and their ends never decrease.  One thread per final site of either scan.  A site of length L at
// s is affected when it touches some edit's core on its own side: s < at + len and s + L > at (a 0-length core: the
// window straddles the junction) -- the first edit k whose core ends behind s decides, found by binary search (dense
// clusters have many edits).  Its window maps to the other side: inside core k at offset o, to the other core's
// start + o when o < min(ref len, alt len) (else it has no partner); before core k, by the net shift of the edits
// before k.  It is paired when the mapped window fits in the other context; a paired window is re-scored there with
// the reference's arithmetic (exact_raw, cscore.c:341-389):
//   ref-list site:  effect 1 (loss) or 3 (both, the alt window passes too);
//   alt-list site:  effect 2 (gain) only when the ref window fails -- else the ref list already has the row.
// The alt list may leave a passing pair to the ref list only because a paired pair of windows is affected on both
// sides or on neither: both windows are placed by the same edit k (the map keeps a start in the same stretch or at the
// same core offset), and both reach core k exactly when s + L passes its start on that side.  The tests' oracle
// derives the rows without this invariant.
// An unpaired site has no window on the other allele: effect 5 (loss) or 6 (gain), the other score NaN, other start
// -1 (row_other == nullptr: not recorded).  Rows are appended (order restored by the sort on row_key = context | motif | own-side start | strand bit
// [| side bit]).  With several edits per context the two sides' coordinates diverge and a ref row and an alt row can
// share (start, strand); the side bit (side_bits = 1) then keeps their keys apart.  With one edit at most one side
// has unpaired windows and no two rows share (start, strand), so side_bits = 0 leaves the single-allele keys as they
// were.
// ---------------------------------------------------------------------------------------------
struct VariantSide {
    SeqView seq;                     // this list's contexts
    const uint64_t *key;             // final sites of the scan of `seq` (motif in the key's motif field)
    const int32_t *seq_idx, *start;
    const int8_t *strand;
    const double *score;
    const int32_t *at, *len;         // this side's edit cores
    int64_t n;
    int key_shift;
};

__device__ __forceinline__ bool site_predicate(const MotifView &M, uint32_t m, double raw, double &score) {
    score = __ddiv_rn(raw, __ldg(M.max_raw + m));                        // cscore.c:357,374
    return __dsub_rn(score, __ldg(M.cutoff + m)) >= -1e-10;              // cscore.c:358,375
}

__global__ void __launch_bounds__(256)
variant_rows_kernel(VariantSide R, VariantSide A, MotifView M, const int64_t *__restrict__ edit_off, int motif_bits,
                    int start_bits, int side_bits, unsigned long long *__restrict__ n_rows, uint64_t *__restrict__ row_key,
                    int32_t *__restrict__ row_idx, double *__restrict__ row_ref, double *__restrict__ row_alt,
                    int8_t *__restrict__ row_eff, int32_t *__restrict__ row_other) {
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R.n + A.n) return;
    const bool from_ref = t < R.n;
    const VariantSide &S = from_ref ? R : A;
    const VariantSide &O = from_ref ? A : R;
    const int64_t i = from_ref ? t : t - R.n;
    const uint32_t m = site_motif(S.key[i], S.key_shift);
    const int32_t s = S.seq_idx[i], st = S.start[i];
    const int L = __ldg(M.len + m);
    int64_t lo = edit_off ? __ldg(edit_off + s) : s, hi = edit_off ? __ldg(edit_off + s + 1) : s + 1;
    const int64_t e1 = hi;
    while (lo < hi) {                                                    // the first edit whose core ends behind st
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(S.at + mid) + __ldg(S.len + mid) > st) hi = mid; else lo = mid + 1;
    }
    if (lo == e1) return;                                                // behind every core
    const int32_t at = __ldg(S.at + lo), oat = __ldg(O.at + lo);
    if (at >= st + L) return;                                            // the window does not touch a changed base
    int32_t ost;                                                         // the window's start on the other side
    bool paired = true;
    if (st >= at) {                                                      // inside core lo
        paired = st - at < min(__ldg(S.len + lo), __ldg(O.len + lo));
        ost = oat + (st - at);
    } else {                                                             // in the shared stretch before core lo
        ost = st + (oat - at);
    }
    paired = paired && ost + L <= __ldg(O.seq.len + s);
    const int rev = S.strand[i] == 2;
    double other = __longlong_as_double(0x7ff8000000000000ll);           // NaN: no window on the other allele
    bool other_hit = false;
    if (paired) {
        const double *pw = M.pwm + 4 * (int64_t) __ldg(M.col_off + m);
        other_hit = site_predicate(M, m, exact_raw(O.seq, pw, L, __ldg(O.seq.poff + s) + ost, rev), other);
        if (!from_ref && other_hit) return;                              // a site on both alleles: the ref list's row
    }
    const unsigned long long slot = atomicAdd(n_rows, 1ull);
    row_key[slot] = (((((uint64_t) s << motif_bits | m) << start_bits | (uint64_t) st) << 1 | (uint64_t) rev)
                     << side_bits) | (uint64_t) (from_ref ? 0 : side_bits);
    row_idx[slot] = (int32_t) slot;
    row_ref[slot] = from_ref ? S.score[i] : other;
    row_alt[slot] = from_ref ? other : S.score[i];
    row_eff[slot] = (int8_t) ((from_ref ? (other_hit ? 3 : 1) : 2) | (paired ? 0 : 4));
    if (row_other) row_other[slot] = paired ? ost : -1;
}

// Sorted row keys + the permutation -> the row arrays in order.
__global__ void __launch_bounds__(256)
variant_gather_kernel(const uint64_t *__restrict__ key, const int32_t *__restrict__ idx, int64_t n, int motif_bits,
                      int start_bits, int side_bits, const double *__restrict__ ref_in, const double *__restrict__ alt_in,
                      const int8_t *__restrict__ eff_in, const int32_t *__restrict__ other_in, int32_t *__restrict__ allele,
                      int32_t *__restrict__ motif, int32_t *__restrict__ start, int8_t *__restrict__ strand,
                      double *__restrict__ ref_out, double *__restrict__ alt_out, int8_t *__restrict__ eff_out,
                      int32_t *__restrict__ other_out) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = key[i] >> side_bits;
    const int32_t j = idx[i];
    allele[i] = (int32_t) (k >> (motif_bits + start_bits + 1));
    motif[i] = (int32_t) ((k >> (start_bits + 1)) & ((1ull << motif_bits) - 1ull));
    start[i] = (int32_t) ((k >> 1) & ((1ull << start_bits) - 1ull));
    strand[i] = (int8_t) ((k & 1ull) + 1);
    ref_out[i] = ref_in[j];
    alt_out[i] = alt_in[j];
    eff_out[i] = eff_in[j];
    if (other_out) other_out[i] = other_in[j];
}

}  // namespace msb
