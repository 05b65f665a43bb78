// prefilter_tc.cuh -- tensor-core prefilter (tcgen05.mma kind::f8f6f4, sm_100a).
//
// The scan's first stage: emit a SUPERSET of the windows the reference
// accepts (cscore.c:340-389); the fp64 exact stage decides.  Formulation:
//
//     D[128 windows x 256 motif-strands] = A[128 x K] * B[256 x K]^T,   K = 4 * Lpad  (e4m3 x e4m3 -> f16)
//
//   A  the one-hot sequence, never materialised as a matrix: shared memory holds a stream of
//      4 bytes per base (e4m3 1.0 in the byte of the base's code, all zero for a non-ACGT base);
//      row r of A is the stream at byte offset 16 r, the window starting 4 bases after row r-1's.
//      In the no-swizzle K-major canonical layout ((8,m),2):((16 B,SBO),LBO) that is SBO = 128 B,
//      LBO = 16 B -- overlapping rows behind one descriptor.  Four copies of the stream shifted
//      by 0..3 bases give the windows at every start.
//   B  per (motif, strand) column the quantised "budget minus deficit" entries
//          e[b][c] = RU_e4m3( beta - s * (colmax_c - V[b][c]) ),   sum_c beta = s * (colmax_sum - T) + margin
//      so that  raw >= T  implies  sum_c e[b_c][c] >= margin > 0: the candidate test is the
//      accumulator's sign bit.  The products are exact (1.0 x e4m3); each K = 32 step adds its
//      exact partial sum to the f16 accumulator with one round-to-nearest (measured,
//      profiles/r1_tc_toeplitz.txt).  For a window with sum >= 0 every partial sum lies in
//      [-C, C], C = L * beta <= 512, so the <= 4 roundings cost <= 4 * 0.125 and the margin C/64
//      >= 5 keeps the sign.  f16 accumulators are read back two per register (.pack::16b), which
//      halves the epilogue's ALU work; the TMEM read itself costs the same as f32.
//
// One CTA per SM, warp-specialised: warp 0 issues the MMAs, warps 1-3 expand packed codes into
// the one-hot streams (3-slot ring), warps 4-19 (two sets of 8, one per 256-column TMEM buffer)
// read the accumulators back, AND-reduce the sign bits and, on the rare clear sign, store one
// 16-byte candidate record per lane and chunk ("Candidate emission" below).
#pragma once
#include "common.cuh"

// Compile-time experiment switch (bench_micro/tc_ablate.sh builds one library per value; results in
// profiles/): 0 = product, 1 = no candidate emission, 2 = no accumulator scan either, 3 = no TMEM
// read-back either (tensor pipe alone), 8 = records stored without computing the flag words,
// 9 = flag words computed but nothing stored, 10 = sign scan + branch only (a hit just counts), 11 = sign scan, no branch (predicated count).  Anything but 0 gives
// wrong results by design.
#ifndef MSB_TC_EXP
#define MSB_TC_EXP 0
#endif

namespace msb {

constexpr int kTcTileBases = 512;                       // window starts per position tile
constexpr int kTcStreamBases = kTcTileBases + 32;       // + halo for the longest motif
constexpr int kTcStreamBytes = kTcStreamBases * 4;      // 2176 B per shifted copy
constexpr int kTcSlotBytes = 4 * kTcStreamBytes;        // 8704 B
constexpr int kTcSlots = 3;
constexpr int kTcIgnoreOff = kTcSlots * kTcSlotBytes;   // 26112: 3 x 16 ignore words
constexpr int kTcBOff = 27 * 1024;                      // B tiles start here (1024-aligned)
constexpr int kTcUnitBytes = 8192;                      // one K=32 step of a 256-column tile
constexpr int kTcMaxUnits = 24;                         // 8 KB K-steps of B per batch (192 KB of shared memory)
constexpr int kTcMaxTiles = kTcMaxUnits;                // tiles per batch
constexpr int kTcCols = 256;                            // motif-strand columns per tile
constexpr int kTcEpiWarps = 16;                         // two sets of 8: set g reads the units that land in TMEM buffer g
constexpr int kTcProducerWarps = 3;                     // warps 1-3 expand the one-hot streams
constexpr int kTcThreads = (4 + kTcEpiWarps) * 32;      // 640 threads x 96 registers
constexpr int kTcWarpCols = 128;                        // accumulator columns one epilogue warp reads per unit
constexpr int kTcSmemBytes = kTcBOff + kTcMaxUnits * kTcUnitBytes;   // dynamic shared memory of the kernel
constexpr int kTcLanesPerCta = kTcEpiWarps * 32;        // epilogue lanes, each with its own candidate-record buffer
constexpr int kTcStaticSmemReserve = 1024;             // static __shared__ (barriers) + alignment slack
// Warp roles.  MSB_TC_ISSUER_LAST = 1: epilogue warps 0-15, MMA issuer warp 16, producers 17-19 (the issuer and the
// producers are the highest warp ids of their sub-partitions); 0: issuer 0, producers 1-3, epilogue 4-19.
#ifndef MSB_TC_ISSUER_LAST
#define MSB_TC_ISSUER_LAST 0
#endif
constexpr int kTcIssuerWarp = MSB_TC_ISSUER_LAST ? kTcEpiWarps : 0;
constexpr int kTcFirstProducer = kTcIssuerWarp + 1;
constexpr int kTcFirstEpi = MSB_TC_ISSUER_LAST ? 0 : 4;

struct TcBatch {
    uint32_t n_tiles;
    uint32_t b_off;                  // byte offset of the batch's tiles in the global B buffer
    uint32_t b_bytes;
    uint32_t first_tile;             // global tile index of the batch's first tile (col_info row)
    uint8_t ks[kTcMaxTiles];         // K steps (of 32 = 8 bases) per tile
    uint8_t unit_off[kTcMaxTiles];   // tile start within the batch, in 8 KB units
};

struct TcParams {
    SeqView seq;
    const uint8_t *btab;       // all tiles: [ks][kchunk16 (2)][column (256)][16 B]
    TcBatch batch;
    int32_t lmax_all;
    int32_t emit_dirty;
    int32_t any_zero_hit;
    int64_t pos_lo, pos_hi;    // only windows starting at packed positions [pos_lo, pos_hi) are scored (range scans)
    uint4 *cand;               // candidate records: buffer of epilogue lane g (= (CTA * 16 + epilogue warp) * 32 + lane) at cand + g * cand_cap
    int64_t cand_cap;          // records per lane buffer
    uint32_t *lane_count;      // [grid * kTcLanesPerCta] records written by each lane so far (carried across launches)
    int64_t *dirty;
    int64_t dirty_cap;
    unsigned long long *counters;   // [1] dirty positions (the record totals are reduced from lane_count by lane_totals_kernel)
    long long *prof;           // optional [grid][16] cycle counters (msb_ctx_set_option(ctx, "tc_prof", 1)); nullptr = off
};

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_f8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// K-major, no swizzle (version 1 descriptor): start address, K-chunk byte offset, 8-row-group byte offset
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t) ((addr & 0x3FFFFu) >> 4) | ((uint64_t) (lbo >> 4) << 16) | ((uint64_t) (sbo >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

#define MSB_TC_LD32(r, addr)                                                                        \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                          \
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"                          \
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"        \
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),  \
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), \
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), \
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]) \
                 : "r"(addr))

#define MSB_TC_LD32P(r, addr)                                                                       \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.pack::16b.x32.b32 "                                \
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"                          \
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"        \
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),  \
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), \
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), \
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]) \
                 : "r"(addr))

__device__ __forceinline__ uint32_t and8(const uint32_t (&r)[32], int g) {
    return (r[8 * g] & r[8 * g + 1] & r[8 * g + 2]) & (r[8 * g + 3] & r[8 * g + 4] & r[8 * g + 5]) & (r[8 * g + 6] & r[8 * g + 7]);
}

// Candidate emission.  A unit's accumulators are in registers when its TMEM buffer is released, but
// a warp cannot start on its next unit before it is done with this one, and a set of eight warps
// recycles a buffer only when all eight have read it.  With ~0.3 candidates per warp and unit nearly
// every unit has SOME warp on the rare path, so whatever the rare path costs is paid by the tensor
// pipe.  Measured with bench_micro/tc_ablate.sh (profiles/r1_c_ablation.txt): 3.9 ms with emission
// compiled out; 6.3-6.8 ms with every variant that staged keys in shared memory from the epilogue
// warps (per-lane slots + out-of-line decode, a warp-uniform ballot path, pre-reserved blocks), and
// 7-13 ms with a shared-memory dump queue drained by a decoder warp: shared memory is ~75 % busy
// feeding the tensor core, so anything that makes round trips through it on the rare path is slow,
// and so is anything that waits for an atomic.  What is left is register-only:
// a lane that sees a clear sign bit in its 64-column chunk folds the chunk's 64 sign bits into two
// words (16 PRMT in sign-replication mode + 16 LOP3) and stores ONE 16-byte record
// {position, first column, 64 flag bits} to ITS OWN buffer in global memory: no shared memory, no
// atomic, no vote, nothing to wait for.  The exact stage expands the flag bits
// (exact_records_kernel, one warp per lane buffer); lane_totals_kernel reduces the per-lane counts.
//
// Record: x = position bits 0..31, y = position bits 32..40 | first column (tile * 256 + column) << 9,
//         z / w = flag words of columns +0..31 / +32..63: within a word, bit 8 b + k <=> column 4 k + b.
__device__ __forceinline__ void st_global_v4(uint4 *p, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ unsigned long long atom_add_global(unsigned long long *p, unsigned long long v) {
    unsigned long long old;
    asm volatile("atom.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
    return old;
}
__device__ __forceinline__ void st_global(uint64_t *p, uint64_t v) {
    asm volatile("st.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// prmt.b32 with selector 0xFDB9: bytes 1 and 3 of x, then bytes 1 and 3 of y, each replaced by its
// sign bit replicated over the byte (selector nibble msb = sign mode): the signs of the four f16
// accumulators of (x, y), one per byte.
__device__ __forceinline__ uint32_t half_signs(uint32_t x, uint32_t y) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, 0xFDB9;" : "=r"(d) : "r"(x), "r"(y));
    return d;
}
// flag word of 16 registers = 32 columns: bit 8 b + k set <=> accumulator 4 k + b has a clear sign
__device__ __forceinline__ uint32_t flag_word(const uint32_t (&r)[32], int half) {
    uint32_t f = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) f |= ~half_signs(r[16 * half + 2 * k], r[16 * half + 2 * k + 1]) & (0x01010101u << k);
    return f;
}

struct LaneOut {
    uint4 *buf;        // this lane's record buffer
    uint32_t n;        // records written (may exceed the capacity: the host then retries with a larger one)
};

// One packed 64-column load of this lane's window: r[j] holds columns col0 + 2j (low half) and
// col0 + 2j + 1 (high half) of the window at packed position p.
__device__ __forceinline__ void scan_chunk(const TcParams &P, LaneOut &out, const uint32_t (&r)[32], bool live,
                                           uint32_t col0, int64_t p) {
    constexpr uint32_t M = 0x80008000u;
    const uint32_t g_lo = and8(r, 0) & and8(r, 1), g_hi = and8(r, 2) & and8(r, 3);
    bool hit = live && ((g_lo & g_hi) & M) != M;
#if MSB_TC_EXP >= 1 && MSB_TC_EXP <= 3
    hit = false;
#endif
#if MSB_TC_EXP == 11
    out.n += hit ? 1u : 0u;   // ablation: the sign scan without any branch
    return;
#endif
    if (hit) {   // divergent, rare; usually one lane and one half: only that half's flag word is computed
#if MSB_TC_EXP == 10
        out.n++;     // ablation: the sign scan and the branch, nothing else
        return;
#endif
        uint32_t z = 0, w = 0;
#if MSB_TC_EXP != 8
        if ((g_lo & M) != M) z = flag_word(r, 0);
        if ((g_hi & M) != M) w = flag_word(r, 1);
#endif
#if MSB_TC_EXP == 9
        out.n += (z ^ w) & 1u;   // ablation: flags computed, nothing stored
        return;
#endif
        if ((int64_t) out.n < P.cand_cap)
            st_global_v4(out.buf + out.n, (uint32_t) p, (uint32_t) ((uint64_t) p >> 32) | (col0 << 9), z, w);
        out.n++;
    }
}

// 32-bit shared-memory addresses of the barriers, computed once per thread.
struct TcBars {
    uint32_t stream_full, stream_empty, tmem_full, tmem_empty;   // address of element 0; 8 B stride
};

__device__ __forceinline__ void mbar_wait_a(uint32_t addr, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t addr) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// descriptor = {lo, hi}: lo = start address >> 4 | LBO >> 4 << 16, hi = SBO >> 4 | version 1 << 14
__device__ __forceinline__ void umma_f8_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                             uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi),
        "r"(idesc), "r"(acc)
        : "memory");
}

}  // namespace tc

// Warp roles: 0 MMA issuer, 1-3 producers, 4-19 epilogue (TMEM lane quarter = warp % 4, column
// share = (warp - 4) / 4).  The scheduler favours the highest warp id of a sub-partition: the
// epilogue warps carry the per-unit critical path, the others mostly poll barriers.
template <bool kProf>
__global__ void __launch_bounds__(kTcThreads, 1)
prefilter_tc_kernel(const __grid_constant__ TcParams P) {
    using namespace tc;
    // cycle counter reads exist only in the profiling instantiation (MSB_TC_PROF=1)
    auto now = [] { return kProf ? clock64() : 0ll; };
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *s_stream = smem;
    uint32_t *s_ignore = reinterpret_cast<uint32_t *>(smem + kTcIgnoreOff);
    uint8_t *s_b = smem + kTcBOff;
    __shared__ uint64_t bar_stream_full[kTcSlots], bar_stream_empty[kTcSlots], bar_tmem_full[2], bar_tmem_empty[2];
    __shared__ uint32_t s_tmem_base;
    __shared__ uint32_t s_skip[kTcSlots];
    __shared__ uint2 s_tile[kTcMaxTiles];   // per tile: B descriptor low word, K steps

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const SeqView &S = P.seq;
    // position tiles [pt_first + blockIdx.x, pt_end) in steps of gridDim.x
    const int64_t pt_first = P.pos_lo / kTcTileBases + blockIdx.x;
    const int64_t n_ptiles = (P.pos_hi + kTcTileBases - 1) / kTcTileBases;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kTcSlots; i++) { mbar_init(&bar_stream_full[i], kTcProducerWarps); mbar_init(&bar_stream_empty[i], 1 + kTcEpiWarps); }
        for (int i = 0; i < 2; i++) { mbar_init(&bar_tmem_full[i], 1); mbar_init(&bar_tmem_empty[i], kTcEpiWarps / 2); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < P.batch.n_tiles) {
        const uint32_t bt = smem_u32(s_b) + (uint32_t) P.batch.unit_off[threadIdx.x] * kTcUnitBytes;
        s_tile[threadIdx.x] = make_uint2(((bt & 0x3FFFFu) >> 4) | ((4096u >> 4) << 16), P.batch.ks[threadIdx.x]);
    }
    if (warp == kTcIssuerWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tmem_base)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    {   // the batch's B tiles -> shared memory, then visible to the async (tensor core) proxy
        const uint4 *src = reinterpret_cast<const uint4 *>(P.btab + P.batch.b_off);
        uint4 *dst = reinterpret_cast<uint4 *>(s_b);
        const uint32_t n16 = P.batch.b_bytes >> 4;
        for (uint32_t i = threadIdx.x; i < n16; i += kTcThreads) dst[i] = __ldg(src + i);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = s_tmem_base;
    const uint32_t NT = P.batch.n_tiles;
    TcBars B;
    B.stream_full = smem_u32(&bar_stream_full[0]);
    B.stream_empty = smem_u32(&bar_stream_empty[0]);
    B.tmem_full = smem_u32(&bar_tmem_full[0]);
    B.tmem_empty = smem_u32(&bar_tmem_empty[0]);

    if (warp == kTcIssuerWarp) {
        // ---- MMA issuer: the whole warp runs the loop (uniform values), one elected lane issues ----
        // D = F16 (0 << 4), A = B = E4M3 (0), both K-major, N = 256 (>> 3 at bit 17), M = 128 (>> 4 at bit 24)
        const uint32_t idesc = ((uint32_t) (kTcCols >> 3) << 17) | ((uint32_t) (128 >> 4) << 24);
        const uint32_t desc_hi = (128u >> 4) | (1u << 14);                 // SBO = 128 B, descriptor version 1
        const uint32_t a_lo0 = ((smem_u32(s_stream) & 0x3FFFFu) >> 4) | ((16u >> 4) << 16);   // LBO = 16 B
        uint32_t u = 0, it = 0;
        long long t_ws = 0, t_we = 0, t_is = 0;
        const long long t_begin = now();
        for (int64_t t = pt_first; t < n_ptiles; t += gridDim.x, it++) {
            const uint32_t slot = it % kTcSlots;
            long long c0 = now();
            mbar_wait_a(B.stream_full + 8 * slot, (it / kTcSlots) & 1);
            t_ws += now() - c0;
            fence_after();
            {
                const uint32_t skipmask = s_skip[slot];   // bit s: no live window starts at a position = s (mod 4) in this tile
#pragma unroll 1
                for (uint32_t s = 0; s < 4; s++) {
                    if ((skipmask >> s) & 1u) continue;
                    const uint32_t a_lo = a_lo0 + ((slot * kTcSlotBytes + s * kTcStreamBytes) >> 4);
                    uint2 tile = s_tile[0];
#pragma unroll 1
                    for (uint32_t nt = 0; nt < NT; nt++, u++) {
                        const uint2 cur = tile;
                        if (nt + 1 < NT) tile = s_tile[nt + 1];     // next tile's descriptor while we wait
                        const uint32_t buf = u & 1;
                        c0 = now();
                        mbar_wait_a(B.tmem_empty + 8 * buf, ((u >> 1) & 1) ^ 1);
                        const long long c1 = now();
                        t_we += c1 - c0;
                        fence_after();
                        if (elect_one()) {
                            const uint32_t d = tmem + buf * kTcCols;
                            umma_f8_lohi(d, a_lo, desc_hi, cur.x, desc_hi, idesc, 0);
                            if (cur.y > 1) umma_f8_lohi(d, a_lo + 2, desc_hi, cur.x + 512, desc_hi, idesc, 1);
                            if (cur.y > 2) umma_f8_lohi(d, a_lo + 4, desc_hi, cur.x + 1024, desc_hi, idesc, 1);
                            if (cur.y > 3) umma_f8_lohi(d, a_lo + 6, desc_hi, cur.x + 1536, desc_hi, idesc, 1);
                            umma_commit_a(B.tmem_full + 8 * buf);
                        }
                        __syncwarp();
                        const long long c4 = now();
                        t_is += c4 - c1;
                        if (kProf && P.prof && blockIdx.x == 0 && lane == 0 && u >= 2000 && u < 2012) {
                            long long *o = P.prof + gridDim.x * 16 + (u - 2000) * 8;
                            o[0] = c1; o[1] = c4;
                        }
                    }
                }
            }
            if (elect_one()) umma_commit_a(B.stream_empty + 8 * slot);   // fires when the MMAs that read the slot are done
            __syncwarp();
        }
        if (kProf && P.prof && lane == 0) {
            long long *o = P.prof + blockIdx.x * 16;
            o[0] = now() - t_begin; o[1] = t_ws; o[2] = t_we; o[3] = t_is; o[4] = u;
        }
    } else if (warp >= kTcFirstProducer && warp < kTcFirstProducer + kTcProducerWarps) {
        // ---- producers: packed codes -> 4 shifted one-hot streams, ignore bits, dirty windows -----
        const int tid_p = (warp - kTcFirstProducer) * 32 + lane;
        const uint32_t horizon = P.lmax_all >= 32 ? 0xffffffffu : ((1u << P.lmax_all) - 1u);
        uint32_t it = 0;
        for (int64_t t = pt_first; t < n_ptiles; t += gridDim.x, it++) {
            const uint32_t slot = it % kTcSlots;
            mbar_wait_a(B.stream_empty + 8 * slot, ((it / kTcSlots) & 1) ^ 1);
            const int64_t tile_start = t * kTcTileBases;
            uint32_t *dst = reinterpret_cast<uint32_t *>(s_stream + slot * kTcSlotBytes);
            for (int a = tid_p; a < kTcStreamBases + 3; a += 32 * kTcProducerWarps) {
                const int64_t p = tile_start + a;
                uint32_t word = 0;
                if (p < S.total_packed) {
                    const uint32_t code = (__ldg(S.codes + (p >> 4)) >> ((p & 15) * 2)) & 3u;
                    const uint32_t isn = (__ldg(S.nmask + (p >> 5)) >> (p & 31)) & 1u;
                    word = isn ? 0u : (0x38u << (8 * code));   // e4m3 1.0 in the byte of the base
                }
#pragma unroll
                for (int s = 0; s < 4; s++) {
                    const int i = a - s;
                    if (i >= 0 && i < kTcStreamBases) dst[s * kTcStreamBases + i] = word;
                }
            }
            if (warp == kTcFirstProducer) {
                uint32_t ign = 0xffffffffu;
                if (lane < 16) {
                    const int64_t q0 = tile_start + lane * 32;
                    // blocks wholly outside the scanned range are never looked up: behind pos_hi the owner
                    // table may not be written yet (msb_scan_ascii encodes slice k + 1 after this launch)
                    if (q0 < S.total_packed && q0 < P.pos_hi && q0 + 32 > P.pos_lo) {
                        const int64_t blk = q0 >> 5;
                        const int64_t s = __ldg(S.blk_seq + blk);
                        const int64_t j0 = q0 - __ldg(S.poff + s);
                        const int64_t left = (int64_t) __ldg(S.len + s) - j0;
                        const int nvalid = left <= 0 ? 0 : (left >= 32 ? 32 : (int) left);
                        uint32_t valid = nvalid >= 32 ? 0xffffffffu : ((1u << nvalid) - 1u);
                        if (S.limit) {   // windows may only start at the first limit[s] positions of the sequence
                            const int64_t lim = (int64_t) __ldg(S.limit + s) - j0;
                            valid &= lim >= 32 ? 0xffffffffu : (lim <= 0 ? 0u : ((1u << (int) lim) - 1u));
                        }
                        // range scans: starts outside [pos_lo, pos_hi) belong to another call
                        if (q0 < P.pos_lo) valid &= P.pos_lo - q0 >= 32 ? 0u : ~((1u << (int) (P.pos_lo - q0)) - 1u);
                        if (q0 + 32 > P.pos_hi) valid &= P.pos_hi <= q0 ? 0u : ((1u << (int) (P.pos_hi - q0)) - 1u);
                        const uint64_t m64 = ((uint64_t) __ldg(S.nmask + blk + 1) << 32) | __ldg(S.nmask + blk);
                        const uint64_t m64hi = (uint64_t) __ldg(S.nmask + blk + 2);   // bases 64..95 (zero padding behind the set)
                        // a dirty window is dropped here only when EVERY base any motif can see is N (then every
                        // motif scores exactly 0, cscore.c:346): for motifs longer than the 32-base horizon that
                        // takes the longest motif's length (<= 64), not the horizon
                        const uint64_t span = P.lmax_all >= 64 ? ~0ull : ((1ull << P.lmax_all) - 1ull);
                        uint32_t dirtym = 0, emitm = 0;
#pragma unroll 1
                        for (int k = 0; k < 32; k++) {
                            const uint32_t bits = (uint32_t) (m64 >> k) & horizon;
                            // bases behind the sequence's end do not exist: a motif that would reach them has no
                            // window here (cscore.c:340), so for the all-N test they count as N
                            const int64_t rem = left - k;
                            const uint64_t beyond = rem >= 64 ? 0ull : (rem <= 0 ? ~0ull : (~0ull << rem));
                            const uint64_t wide = ((m64 >> k) | (k ? m64hi << (64 - k) : 0ull) | beyond) & span;
                            dirtym |= (bits != 0 ? 1u : 0u) << k;
                            emitm |= ((bits != 0 && !(wide == span && !P.any_zero_hit)) ? 1u : 0u) << k;
                        }
                        ign = dirtym | ~valid;
                        if (P.emit_dirty) {
                            // windows that touch a non-ACGT base go to the exact kernel directly
                            uint32_t e = emitm & valid;
                            while (e) {
                                const int k = __ffs(e) - 1;
                                e &= e - 1;
                                const unsigned long long sl = atom_add_global(P.counters + 1, 1ull);
                                if ((int64_t) sl < P.dirty_cap) st_global(reinterpret_cast<uint64_t *>(P.dirty) + sl, (uint64_t) (q0 + k));
                            }
                        }
                    }
                    s_ignore[slot * 16 + lane] = ign;
                }
                // shift s of the tile holds the windows starting at positions = s (mod 4): when all of them are
                // ignored (N runs, padding, a start limit that leaves only offset 0 of each sequence) its
                // MMAs are not issued at all
                uint32_t skipmask = 0;
#pragma unroll
                for (int sft = 0; sft < 4; sft++)
                    skipmask |= (__all_sync(0xffffffffu, (ign | ~(0x11111111u << sft)) == 0xffffffffu) ? 1u : 0u) << sft;
                if (lane == 0) s_skip[slot] = skipmask;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive_a(B.stream_full + 8 * slot);
        }
    } else {
        // ---- epilogue: warp reads TMEM lanes 32 q .. 32 q + 31 (its 32 windows), 128 of the 256 columns
        const int ew = warp - kTcFirstEpi;       // epilogue warp 0..15; kTcFirstEpi is a multiple of 4, so ew % 4 == warp % 4
        const int q = warp & 3, h = (ew >> 2) & 1, set = ew >> 3;
        const int row = q * 32 + lane;
        LaneOut out;
        const size_t lane_id = ((size_t) blockIdx.x * kTcEpiWarps + ew) * 32 + lane;
        out.buf = P.cand + lane_id * (size_t) P.cand_cap;
        out.n = P.lane_count[lane_id];
        const uint32_t taddr0 = tmem + set * kTcCols + h * kTcWarpCols + ((uint32_t) (q * 32) << 16);
        const uint32_t colid0 = P.batch.first_tile * kTcCols + h * kTcWarpCols;
        uint32_t u = 0, it = 0;
        long long t_wf = 0, t_ld = 0, t_pr = 0, t_wsf = 0, t_slow = 0, n_slow = 0;
        for (int64_t t = pt_first; t < n_ptiles; t += gridDim.x, it++) {
            const uint32_t slot = it % kTcSlots;
            const long long cs = now();
            mbar_wait_a(B.stream_full + 8 * slot, (it / kTcSlots) & 1);
            t_wsf += now() - cs;
            const uint32_t skipmask = s_skip[slot];
            const uint32_t ign4 = (s_ignore[slot * 16 + (row >> 3)] >> ((row & 7) * 4)) & 0xFu;
            __syncwarp();
            if (lane == 0) mbar_arrive_a(B.stream_empty + 8 * slot);
            if (skipmask == 0xFu) continue;
            const int64_t tile_start = t * kTcTileBases;
            // units of this tile, in the issuer's order: for every shift that is not skipped, the NT tiles.
            // Unit u + v lands in TMEM buffer (u + v) & 1; this warp set reads the ones in buffer `set`.
            uint32_t act = 0, n_act = 0;                       // act: the active shifts, 2 bits each
            for (uint32_t sft = 0; sft < 4; sft++)
                if (!((skipmask >> sft) & 1u)) { act |= sft << (2 * n_act); n_act++; }
            const uint32_t n_units = n_act * NT;
            const uint32_t v0 = ((uint32_t) set ^ u) & 1u;
            uint32_t ai = 0, nt = v0;
            while (nt >= NT) { nt -= NT; ai++; }
#pragma unroll 1
            for (uint32_t v = v0; v < n_units; v += 2) {
                const uint32_t sh = (act >> (2 * ai)) & 3u;
                const uint32_t uu = u + v;
                const bool live = !((ign4 >> sh) & 1u);
                const int64_t p = tile_start + 4 * row + sh;
                const uint32_t colid = colid0 + nt * kTcCols;
                const long long c0 = now();
                mbar_wait_a(B.tmem_full + 8 * set, (uu >> 1) & 1);
                const long long c1 = now();
                t_wf += c1 - c0;
                fence_after();
                uint32_t r0[32], r1[32];
#if MSB_TC_EXP != 3
                MSB_TC_LD32P(r0, taddr0);        // columns [0, 64) of this warp's share, two per register
                MSB_TC_LD32P(r1, taddr0 + 64);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#else
                r0[0] = r0[31] = 0;
#endif
                fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_a(B.tmem_empty + 8 * set);   // accumulators are in registers
                const long long c2 = now() + ((r0[0] ^ r0[31]) == 0x12345679u);   // depends on the loaded data
                t_ld += c2 - c1;
                const uint32_t n_before = out.n;
#if MSB_TC_EXP != 2 && MSB_TC_EXP != 3
                scan_chunk(P, out, r0, live, colid, p);
                scan_chunk(P, out, r1, live, colid + 64, p);
#endif
                if (kProf) {
                    const long long c3 = now();
                    t_pr += c3 - c2;
                    if (__any_sync(0xffffffffu, out.n != n_before)) { t_slow += c3 - c2; n_slow++; }
                    if (P.prof && blockIdx.x == 0 && lane == 0 && (ew == 0 || ew == 8) && uu >= 2000 && uu < 2012) {
                        long long *o = P.prof + gridDim.x * 16 + (uu - 2000) * 8;
                        o[2] = c0; o[3] = c1; o[4] = c2; o[5] = c3; o[6] = warp;
                    }
                }
                nt += 2;
                while (nt >= NT) { nt -= NT; ai++; }
            }
            u += n_units;
        }
        P.lane_count[lane_id] = out.n;
        if (kProf && P.prof && ew == 0 && lane == 0) {
            long long *o = P.prof + blockIdx.x * 16;
            o[8] = t_wf; o[9] = t_ld; o[10] = t_pr; o[11] = t_wsf; o[12] = u; o[13] = t_slow; o[14] = n_slow;
        }
    }
    fence_before();
    __syncthreads();
    if (warp == kTcIssuerWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}

}  // namespace msb
