// common.cuh -- shared host/device definitions for libmsb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "msb200.h"

namespace msb {

// ---- limits of the prefilter path ------------------------------------------------------------
constexpr int kMaxFastLen = 32;               // columns the prefilter looks at (the register window of the exact stage)
constexpr int kMaxTcLen = 64;                 // longest motif the prefilter takes (prefiltered on kMaxFastLen columns)
constexpr int kPadBases = 32;                 // every sequence is padded to a multiple of this

// Site key: motif | packed position | strand bit.
// Sorting ascending by this key yields the reference's list order
// (motif, sequence, start, forward before reverse; cscore.c:336-389).
constexpr int kPosBits = 41;                  // packed positions < 2^41 (2.2e12 bases)
constexpr int kMotifShift = kPosBits + 1;
__host__ __device__ inline uint32_t key_rev(uint64_t k) { return (uint32_t) (k & 1); }
// Site keys use the same layout with a per-scan motif shift = (bits of the largest packed position)
// + 1, so the radix sort that orders the sites touches no empty bit range: 37 key bits = 5 passes
// for configs[1] instead of the 52 bits = 7 passes of the fixed layout.
__host__ __device__ inline uint64_t make_site_key(uint32_t motif, int64_t pos, uint32_t rev, int shift) {
    return ((uint64_t) motif << shift) | ((uint64_t) pos << 1) | rev;
}
__host__ __device__ inline uint32_t site_motif(uint64_t k, int shift) { return (uint32_t) (k >> shift); }
__host__ __device__ inline int64_t site_pos(uint64_t k, int shift) { return (int64_t) ((k & ((1ull << shift) - 1)) >> 1); }

// ---- error plumbing --------------------------------------------------------------------------
void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define MSB_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t _e = (call);                                              \
        if (_e != cudaSuccess) return ::msb::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

#define MSB_TRY(call)                 \
    do {                              \
        int _rc = (call);             \
        if (_rc != MSB_OK) return _rc; \
    } while (0)

// Grow-only device buffer.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes);
    void release();
    template <typename T> T *as() const { return (T *) p; }
};

// ---- device-side views -----------------------------------------------------------------------
struct SeqView {
    const uint32_t *codes;   // 2-bit codes, 16 bases per word, base i at bits [2i, 2i+1]; N -> 0
    const uint32_t *nmask;   // 1 bit per base, 32 bases per word; 1 = not A/C/G/T
    const int64_t *poff;     // [n_seqs + 1] packed start of every sequence (multiple of 32)
    const int32_t *len;      // [n_seqs] true length in bases
    const int32_t *blk_seq;  // [total_packed / 32] sequence that owns each 32-base block
    const int32_t *limit;    // [n_seqs] windows may start at positions < limit (<= len); nullptr = len
    int64_t n_seqs;
    int64_t total_packed;    // poff[n_seqs]
};

struct MotifView {
    const double *pwm;       // motif m, column c, row r at pwm[4 * (col_off[m] + c) + r]
    const int32_t *col_off;  // [n_motifs + 1]
    const int32_t *len;      // [n_motifs]
    const double *cutoff;    // [n_motifs]
    const double *max_raw;   // [n_motifs]  cscore.c:36-48
    const float *pwm32;      // the same matrices rounded to fp32, same layout (screening only)
    const float *floor32;    // [n_motifs] an fp32-accumulated raw score below this cannot be a site
    int32_t n_motifs;
};

}  // namespace msb
