// K4 + K5 on the 5th-generation tensor cores: contig x reference distance contraction with a fused candidate-selection
// epilogue, followed by an exact float64 decision kernel.
//
// Replaces learning.knn (reference scripts/learning.py:118-128), the per-contig nearest-centroid loop
// (scripts/phamer.py:251-255 -> learning.closest_to :59-66) and proximity_metric (scripts/phamer.py:198-210).
//
//   d2(a, b) = |a|^2 + |b|^2 - 2 a.b          a = contig features [n, 256], b = reference rows / centroids
//
// Canonical 4-mer features (136 wide) take the same road: a row fills the first 136 operand columns, centred by 1/136, and the
// other 120 columns are exactly zero on both sides, so the contraction kernel is the same and every bound below holds for the
// 136-wide vectors.  Every kernel that reads float64 or count rows takes the width as its template parameter W.
// 5-mer features (1024 plain, 512 canonical) take operands of their own width (OPW<W> = W, NK = W / 64 K-chunks); the query tile
// is then streamed through the ring with the reference blocks instead of staying resident (score_tc_kernel<KN, LIST, NK>).  The
// bound below is stated for any width: |b'|^2 = |b|^2 - 1/W < 1 keeps the three-way split of nbs exact, every scaled centred feature
// lies in (-2^12/W, 2^12) inside the FP16 range, and FP16 rounds 5-mer values (about 4x smaller) with the same relative error, so
// the scale 2^12 stays; only the accumulation allowance grows with the number of MMAs (see eps_acc).
//
// The a.b term is a dense contraction and runs as ONE tcgen05.mma pass (kind::f16, FP32 accumulators in tensor memory) over
// operands that are centred by 1/256 (distances are translation invariant), scaled by 2^12 and rounded to FP16.  FP16 x FP16
// products are exact in FP32, so the only errors are the operand roundings and the FP32 accumulation; both are BOUNDED, per
// (contig, reference) pair, by quantities that are computed exactly when the operands are prepared:
//
//     A = fp16(A~), A~ = 2^12 (a - 1/256)   dA = |A~ - A|_2 , nA = |A|_2          (per contig)
//     B = fp16(B~), B~ = 2^12 (b - 1/256)   dB = |B~ - B|_2 , P  = |B~|_2         (per reference)
//     A~.B~ - A.B = (A~ - A).B~ + A.(B~ - B)         =>   |A~.B~ - acc| <= dA P + nA dB + eps_acc nA (P + dB)
//
// (Cauchy-Schwarz; eps_acc = 2^-16 covers 16 FP32-accumulated MMAs, measured usage of the whole bound <= 0.4.)  The allowance
// is 2^-20 of |A| |B| per accumulating MMA of K = 16 (16x the 2^-24 of one FP32 add, for the tensor core's own accumulation order):
// a sum of m such steps errs by at most m 2^-20 sum_i |A_i B_i| <= m 2^-20 |A| |B|, so with NK K-chunks of 64 (4 NK MMAs)
// eps_acc = NK 2^-18: 2^-16 at 256 (NK = 4), 2^-15 at 512, 2^-14 at 1024 (EPS_ACC_OF).  With
// rho = max_j (dB_j + eps_acc (P_j + dB_j)) / P_j over the reference set this collapses to   err_j <= C_row * P_j  with ONE
// constant per contig row.  The ranking value x_j = 2^23 |b_j - u|^2 - acc_j therefore pins the exact value inside
// [lo_j, up_j] = [x_j - C P_j, x_j + C P_j].  A reference can be one of the k nearest only if lo_j <= (k-th smallest up);
// the epilogue keeps exactly those (they are few: the interval is ~1 % of the distance), straight out of tensor memory, and
// score_decide_kernel reads the vote off them when it is already decided, or re-measures them in float64 by direct
// difference.  Centroid distances that enter tanh((e_n - e_p)/(e_p + e_n)) are always exact float64.  A row whose candidate
// buffer overflows is re-scored exhaustively in float64 (score_fallback_kernel).  The results are therefore those of exact
// arithmetic; the tensor cores only decide WHICH handful of the R references need to be looked at.
//
// Kernel layout (one CTA per SM, persistent over 256-contig tiles, 10 warps):
//   warp 0    TMA producer   A tile (256 contigs x 256 features FP16, 128 KB, SWIZZLE_128B) once per contig tile;
//                            B blocks (128 references x 64 features, 16 KB) through a 4-deep mbarrier ring
//                            (NK > 4: no resident A; every ring stage holds a B block and both 16 KB A halves of its K-chunk)
//   warp 1    MMA issuer     one elected lane: per B block 2 x 4 tcgen05.mma (128x128x16), i.e. two 128-row halves share every
//                            B block, into one of two 2 x 128-column accumulator sets (all 512 TMEM columns);
//                            tcgen05.commit frees the block / publishes the accumulator set
//   warps 2-9 epilogue       thread = contig row = tensor-memory lane.  32 columns per tcgen05.ld (next load in flight while
//                            the current one is scanned): lo_j = fma(-C, P_j, nbs_j - acc_j), running minimum; only when some
//                            lane's minimum beats its threshold are the hits examined (bit mask, then per hit: k smallest
//                            upper bounds in registers + append to the row's candidate buffer in shared memory)
#include <cuda.h>
#include <cuda_fp16.h>
#include <math.h>

#include "score_common.cuh"

namespace phm {

int score_force_fallback = 0;     // option "score_force_fallback": the first pass keeps no candidate, so every row takes the overflow road
                                  // (list pass, or the exhaustive kernels when that is off) -- how the tests reach those kernels
int score_collect_stats = 0;      // option "score_stats": re-measure every candidate and record how much of the bound is used
int score_list_pass = 1;          // option "score_list_pass": 0 = overflowed rows go straight to the exhaustive kernels

namespace tc {

constexpr int KDIM = 256;                 // width of the FP16 operands (plain 4-mers; canonical rows are zero-padded to it)
constexpr int BM = 128, BN = 128, BK = 64;
constexpr int MT = 2 * BM;                // contig rows per CTA tile (two MMA row blocks share every B block)
constexpr int NKC = KDIM / BK;            // 4 K-chunks of 128 bytes
constexpr int NSTAGE = 4;                 // ring of B blocks
constexpr int BLOCK_BYTES = BM * BK * 2;  // 16 KB: 128 rows x 128 B
constexpr int A_BYTES = 2 * NKC * BLOCK_BYTES;          // [half][kc]
constexpr int NEPI = MT;                  // epilogue threads (one per contig row of the tile)
constexpr int CAP_R = 10;                 // candidate slots per row: references
constexpr int CAP_C = 3;                  //                          centroids of one class
constexpr int NENT = CAP_R + 2 * CAP_C;   // 16 entries of 8 bytes per row
constexpr int CAND_BYTES = NEPI * NENT * 8;
constexpr int STG_BYTES = 2 * 2 * BN * 4; // [accumulator set][nbs | P][128 columns] floats
constexpr int BAR_BYTES = 256;
constexpr int SMEM_BYTES = A_BYTES + NSTAGE * BLOCK_BYTES + CAND_BYTES + STG_BYTES + BAR_BYTES;
constexpr int NTHREADS = 64 + NEPI;
constexpr int TMEM_COLS = 512;            // two sets of (2 halves x 128 columns) FP32 accumulators
constexpr float SCALE = (float)PREP_SCALE;  // operands are scaled by 2^12 -> accumulator = 2^24 a'.b'
static_assert(KDIM == PREP_DIM, "score_common.cuh prepares 256-wide rows");
constexpr int LIST_MAX_ROWS = 16384;      // rows the second ("list") tensor-core pass can take (multiple of MT)
constexpr int64_t LIST_POOL = (int64_t)1 << 25;   // most listed references of all such rows together (4 bytes each; the pool is 2048 per
                                                  // possible row up to this); rows that do not fit go to the exhaustive kernels
constexpr uint32_t LIST_NO_ROOM = 0xFFFFFFFFu;
static_assert(LIST_MAX_ROWS % MT == 0, "whole contig tiles");
constexpr double NORM_SCALE = 8388608.0;  // 2^23: ranking value = 2^23 (|b'|^2 - 2 a'.b')
constexpr float PAD_NORM = 3.0e38f;
constexpr double EPS_ACC = 1.0 / 65536.0; // FP32 accumulation allowance relative to |A| |B|
constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);   // F16 x F16 -> F32, K-major
// Seventeenth k-step (round 2): 16 extra K columns turn the accumulator into the LOWER BOUND itself.  A row carries
// (2^10, 2^-1, 2^-12, C16, 0 ...), a reference (-n1, -n2, -n3, P16, 0 ...), where n1 2^10 + n2 2^-1 + n3 2^-12 is the three-way FP16
// split of nbs_j = 2^23 |b'_j|^2 (33 mantissa bits: exact for every float), C16 >= C_row and P16 >= P_j are rounded UP to FP16.  The
// accumulator then holds  S_ij = 2^24 a'_i.b'_j - nbs_j + C16_i P16_j,  and  lo_ij = -S_ij <= x_ij - C_i P_j  is a valid lower bound
// (a little more conservative: both factors were rounded up), up_ij = lo_ij + 2 C16_i P16_j a valid upper bound.  The epilogue is
// a bare maximum over the accumulators: no per-column loads, no subtraction, no multiply-add, no quick reject.
// The extra operands are 128 rows x 32 bytes in the NO-SWIZZLE K-major canonical layout (8 x 16-byte core matrices: row r, K half h
// at (r >> 3) * 256 + h * 128 + (r & 7) * 16), prepared in that order in global memory and brought in by plain bulk copies: the
// block of a reference tile and the two blocks of the contig tile travel together in a fifth slot of the B ring per tile.
constexpr int XK = 16;
constexpr int XBLK_BYTES = BM * XK * 2;   // 4 KB
// 5-mer rows (W = 512, 1024) take operands of their own width: NK = W / 64 K-chunks.  A 256-row A tile is then 256 or 512 KB and
// cannot stay resident, so A is STREAMED: each ring stage carries the reference block and the two 128-row A halves of one K-chunk
// (48 KB), and A is read from L2 once per reference tile.  NK = NKC keeps the resident-A kernel exactly as it is.
template <int W> constexpr int OPW = W <= KDIM ? KDIM : W;           // FP16 operand width of W-wide rows
template <int W> constexpr int NK_OF = OPW<W> / BK;                  // its K-chunks
template <int NK> constexpr bool STREAM_A = NK > NKC;
template <int NK> constexpr int STAGE_BYTES = STREAM_A<NK> ? 3 * BLOCK_BYTES : BLOCK_BYTES;   // [B block][A half 0][A half 1]
template <int NK> constexpr int SMEM_BYTES_OF = (STREAM_A<NK> ? 0 : A_BYTES) + NSTAGE * STAGE_BYTES<NK> + CAND_BYTES + STG_BYTES + BAR_BYTES;
// FP32 accumulation allowance for 4 NK MMAs of K = 16 (2^-20 of |A| |B| per MMA): 2^-16 at NK = 4, 2^-15 at 8, 2^-14 at 16
template <int NK> constexpr double EPS_ACC_OF = (double)NK / 262144.0;
static_assert(SMEM_BYTES_OF<NKC> == SMEM_BYTES && EPS_ACC_OF<NKC> == EPS_ACC, "the 256-wide kernel keeps its layout and bound");
static_assert(SMEM_BYTES_OF<8> <= 232448 && SMEM_BYTES_OF<16> <= 232448, "shared memory budget of one sm_100 CTA (streamed A)");
static_assert(NSTAGE * STAGE_BYTES<16> % 1024 == 0 && (3 * BLOCK_BYTES) % 1024 == 0, "SWIZZLE_128B blocks stay 1024-byte aligned");
constexpr int XBLK_HALVES = XBLK_BYTES / 2;
static_assert(3 * XBLK_BYTES <= BLOCK_BYTES, "the extra operands of a tile fit one ring slot");
__host__ __device__ __forceinline__ int64_t xrow_offset(int64_t row) {      // in halves, K half 0 (K half 1, all zero, is 64 halves further)
    return (row >> 7) * XBLK_HALVES + ((row & 127) >> 3) * 128 + (row & 7) * 8;
}
static_assert(SMEM_BYTES <= 232448, "shared memory budget of one sm_100 CTA");

// ---------------- PTX helpers ----------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ bool elect_one() {                  // true in exactly one lane of a converged warp
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(IDESC), "r"(accumulate), "r"(0u) : "memory");
}
// K-major, SWIZZLE_128B operand tile: rows of 128 bytes, 8-row swizzle atoms 1024 bytes apart
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major), 16-byte units
    d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ float c16_up(float c) { return __half2float(__float2half_ru(c)); }
// K-major, no swizzle: core matrices of 8 rows x 16 bytes; K halves 128 bytes apart (leading offset), 8-row groups 256 bytes apart
__device__ __forceinline__ uint64_t smem_desc_plain(uint32_t addr) {
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(128 >> 4) << 16;           // leading byte offset: next core matrix along K
    d |= (uint64_t)(256 >> 4) << 32;           // stride byte offset: next 8-row group
    d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
    return d;                                  // layout type 0: no swizzle
}
// 32 consecutive accumulator columns of this thread's row; the result registers are valid after tmem_wait_ld()
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}

// ---------------- epilogue building blocks ----------------
// k smallest upper bounds seen so far, ascending; u[K-1] is the row's threshold
template <int K>
__device__ __forceinline__ void upper_insert(float (&u)[K], float v) {       // 2K min/max, branch-free
#pragma unroll
    for (int i = 0; i < K; ++i) {
        const float keep = fminf(u[i], v);
        v = fmaxf(u[i], v);
        u[i] = keep;
    }
}

// Candidate buffer of one row: entries `first` .. `first + CAP - 1` of the thread's 16 slots; entry e of thread t lives at
// cand_addr + e * (NEPI * 8) (cand_addr already holds the thread's 8-byte column, so a warp touches 256 contiguous bytes).
template <int CAP>
__device__ __forceinline__ void cand_prune(uint32_t cand_addr, int first, int &cnt, float limit) {
    int w = 0;
#pragma unroll
    for (int e = 0; e < CAP; ++e) {
        const uint2 ent = lds_v2(cand_addr + (uint32_t)(first + e) * (NEPI * 8));
        if (e < cnt && __uint_as_float(ent.x) <= limit) {
            sts_v2(cand_addr + (uint32_t)(first + w) * (NEPI * 8), ent.x, ent.y);
            ++w;
        }
    }
    cnt = w;
}

template <int CAP>
__device__ __forceinline__ void cand_append(uint32_t cand_addr, int first, int &cnt, uint32_t &flags, float (&drop_lo)[2], float limit,
                                            float lo, int col, int label) {
    if (cnt == CAP) cand_prune<CAP>(cand_addr, first, cnt, limit);
    if (cnt == CAP) {
        // More live candidates than slots.  A labelled (reference) candidate is dropped, but the smallest lower bound dropped
        // per label is remembered: once the scan is over, a dropped label only matters if that bound still reaches the final
        // threshold, and then the vote can still be read off when everything that could be among the k nearest -- kept or
        // dropped -- carries one label (a contig inside a cloud of near-identical references).  Anything else (and any
        // centroid overflow) sends the row to the exhaustive kernels.
        if (label < 0) flags |= 1u;
        else drop_lo[label] = fminf(drop_lo[label], lo);
    } else {
        sts_v2(cand_addr + (uint32_t)(first + cnt) * (NEPI * 8), __float_as_uint(lo), (uint32_t)col);
        ++cnt;
    }
}

__device__ __forceinline__ float pick32(const float (&v)[32], int j) {       // v[j] for a warp-uniform j
    switch (j) {
#define PHM_PICK(i) case i: return v[i];
        PHM_PICK(0) PHM_PICK(1) PHM_PICK(2) PHM_PICK(3) PHM_PICK(4) PHM_PICK(5) PHM_PICK(6) PHM_PICK(7)
        PHM_PICK(8) PHM_PICK(9) PHM_PICK(10) PHM_PICK(11) PHM_PICK(12) PHM_PICK(13) PHM_PICK(14) PHM_PICK(15)
        PHM_PICK(16) PHM_PICK(17) PHM_PICK(18) PHM_PICK(19) PHM_PICK(20) PHM_PICK(21) PHM_PICK(22) PHM_PICK(23)
        PHM_PICK(24) PHM_PICK(25) PHM_PICK(26) PHM_PICK(27) PHM_PICK(28) PHM_PICK(29) PHM_PICK(30)
#undef PHM_PICK
        default: return v[31];
    }
}

__device__ __forceinline__ float max32(const uint32_t (&r)[32]) {
    float g[8];
#pragma unroll
    for (int q = 0; q < 8; ++q)
        g[q] = fmaxf(fmaxf(__uint_as_float(r[4 * q + 0]), __uint_as_float(r[4 * q + 1])), fmaxf(__uint_as_float(r[4 * q + 2]), __uint_as_float(r[4 * q + 3])));
    return fmaxf(fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3])), fmaxf(fmaxf(g[4], g[5]), fmaxf(g[6], g[7])));
}
// 32 accumulator columns of this thread's row (already in registers).  The accumulator IS the negated lower bound (see XK above):
// the chunk's smallest lower bound is minus the largest accumulator, and only if it beats the row's threshold in some lane of the
// warp are the hits looked at, one warp-uniform column at a time.
// INSERT = false: the threshold is already final for these columns (second pass of a two-pass tile), hits are only collected.
template <int K, int CAP, bool INSERT, bool LABELLED>
__device__ __forceinline__ void scan_chunk(const uint32_t (&r)[32], uint32_t p_c, int col_c,
                                           int n_class, float C, uint32_t cand_addr, int first, float (&u)[K], int &cnt,
                                           uint32_t &flags, float (&drop_lo)[2]) {
    const float limit0 = u[K - 1];
    const float m = -max32(r);
    if (!__any_sync(FULL, m <= limit0)) return;
    float lo[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) lo[j] = -__uint_as_float(r[j]);

    // sign of (limit - lo) shifted in column by column: column 0 ends in the top bit, a clear bit is a hit (lo <= limit)
    uint32_t mq[4] = {0u, 0u, 0u, 0u};                   // four independent chains of 8 columns
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) mq[c] = __funnelshift_l(__float_as_uint(limit0 - lo[8 * c + j]), mq[c], 1);
    const uint32_t miss = (mq[0] << 24) | ((mq[1] & 255u) << 16) | ((mq[2] & 255u) << 8) | (mq[3] & 255u);
    const uint32_t hits = __brev(~miss);
    // make room once for the whole warp (one uniform pass) instead of lane by lane inside the loop
    if (__any_sync(FULL, cnt + __popc(hits) > CAP)) cand_prune<CAP>(cand_addr, first, cnt, limit0);
    // Common case: a lane's only hit is its minimum, whose value it already holds -- all such lanes are served at once.
    // Lanes with several hits in the chunk take the column-by-column loop below (warp-uniform column, value picked from the
    // registers by a compile-time switch).
    const int n_hits = __popc(hits);
    if (n_hits == 1) {
        const int j = __ffs(hits) - 1;
        if (m <= u[K - 1] && col_c + j < n_class) {
            const uint32_t pbits = lds_u32(p_c + 4u * j);        // lowest mantissa bit of P carries the reference's label
            if (INSERT) upper_insert<K>(u, fmaf(2.0f * C, __uint_as_float(pbits), m));
            cand_append<CAP>(cand_addr, first, cnt, flags, drop_lo, u[K - 1], m, col_c + j, LABELLED ? (int)(pbits & 1u) : -1);
        }
    }
    // Lanes with several hits in the chunk walk their OWN hit bits (a divergent loop; the values come back from a thread-local copy
    // of the 32 bounds, indexed dynamically).  Round 1 walked the union of all lanes' hit columns warp-uniformly -- up to 32 rounds
    // in the tiles right after the first, where every row still has several hits per chunk -- and that, not the scan, was what kept
    // an accumulator set from going back to the MMA warp.
    uint32_t multi = n_hits > 1 ? hits : 0u;
    if (__any_sync(FULL, multi != 0u)) {
        float lo_mem[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) lo_mem[j] = lo[j];
        while (multi) {
            const int j = __ffs(multi) - 1;
            multi &= multi - 1u;
            const float lo_j = lo_mem[j];
            if (lo_j <= u[K - 1] && col_c + j < n_class) {
                const uint32_t pbits = lds_u32(p_c + 4u * j);
                if (INSERT) upper_insert<K>(u, fmaf(2.0f * C, __uint_as_float(pbits), lo_j));
                cand_append<CAP>(cand_addr, first, cnt, flags, drop_lo, u[K - 1], lo_j, col_c + j, LABELLED ? (int)(pbits & 1u) : -1);
            }
        }
    }
}

// First pass of a two-pass tile: every column's upper bound goes through the branch-free insertion network, so that the
// threshold is already tight when the hits are collected (scan_chunk<.., false> over the same accumulators).
template <int K>
__device__ __forceinline__ void bound_chunk(const uint32_t (&r)[32], uint32_t p_c, float C, float (&u)[K]) {
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const uint4 pp = lds_v4(p_c + 16u * g);
        const float ppv[4] = {__uint_as_float(pp.x), __uint_as_float(pp.y), __uint_as_float(pp.z), __uint_as_float(pp.w)};
#pragma unroll
        for (int i = 0; i < 4; ++i) upper_insert<K>(u, fmaf(2.0f * C, ppv[i], -__uint_as_float(r[4 * g + i])));
    }
}

// One tile (128 columns) of this thread's row: four 32-column loads, the next one in flight while one is scanned.
// TWO_PASS (first reference tile of a contig tile, centroid tiles): thresholds start at +inf there, so nearly every column
// would be a hit; instead all 128 upper bounds go through the insertion network first and the hits are collected in a second
// sweep over the same accumulators (they stay in tensor memory until the set is released).
template <int K, int CAP, bool TWO_PASS, bool LABELLED>
__device__ __forceinline__ void scan_tile(uint32_t taddr, uint32_t p_addr, int col0, int n_class, float C,
                                          uint32_t cand_addr, int first, float (&u)[K], int &cnt, uint32_t &flags, float (&drop_lo)[2]) {
    uint32_t ra[32], rb[32];
    __syncwarp();                                      // tcgen05.ld is .sync.aligned: the warp must be converged
    tmem_ld32_issue(taddr, ra);
    tmem_wait_ld();
    if (TWO_PASS) {
        tmem_ld32_issue(taddr + 32u, rb);
        bound_chunk<K>(ra, p_addr, C, u);
        tmem_wait_ld();
        tmem_ld32_issue(taddr + 64u, ra);
        bound_chunk<K>(rb, p_addr + 128u, C, u);
        tmem_wait_ld();
        tmem_ld32_issue(taddr + 96u, rb);
        bound_chunk<K>(ra, p_addr + 256u, C, u);
        tmem_wait_ld();
        tmem_ld32_issue(taddr, ra);
        bound_chunk<K>(rb, p_addr + 384u, C, u);
        tmem_wait_ld();
    }
    // The four chunks run through TWO copies of the scan code (a rolled loop over chunk pairs), not four.  With four inlined copies the
    // kernel had 15 700 instructions and a fifth of the epilogue's issue slots was lost to instruction fetch (ncu: stall_no_inst 18 %);
    // measured on 1 M contigs x 4510 references: 3.09 -> 2.84 ms.
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        tmem_ld32_issue(taddr + 64u * (uint32_t)h + 32u, rb);
        scan_chunk<K, CAP, !TWO_PASS, LABELLED>(ra, p_addr + 256u * (uint32_t)h, col0 + 64 * h, n_class, C, cand_addr, first, u, cnt, flags, drop_lo);
        __syncwarp();
        tmem_wait_ld();
        if (h == 0) tmem_ld32_issue(taddr + 64u, ra);
        scan_chunk<K, CAP, !TWO_PASS, LABELLED>(rb, p_addr + 256u * (uint32_t)h + 128u, col0 + 64 * h + 32, n_class, C, cand_addr, first, u, cnt,
                                                 flags, drop_lo);
        __syncwarp();
        if (h == 0) tmem_wait_ld();
    }
}

// ---------------- list mode: second pass over the rows whose candidate buffer overflowed ----------------
// After the first pass such a row has a FINAL threshold T (the k-th smallest upper bound among what it kept), so no running
// state is needed: every reference with lo_j <= T is appended to the row's list in global memory, independently per
// reference tile -- which lets (contig tile, reference slice) pairs run on different CTAs.  score_list_decide_kernel then
// measures the listed references exactly.  The pass runs twice: first it only COUNTS the references under each threshold, a
// prefix sum (tc_list_scan_kernel) gives every row its range in one shared pool, then the same pass FILLS the ranges
// (cols != nullptr).  Lists are usually short (the interval is ~1 % of the distance) but a contig far from every reference
// can have thousands of references inside it; only rows that do not fit in the pool go to the exhaustive kernels.
__device__ __forceinline__ void list_chunk(const uint32_t (&r)[32], int col_c, int n_class, float T, uint32_t *cnt, uint32_t *cols) {
    if (!__any_sync(FULL, -max32(r) <= T)) return;
    uint32_t hits = 0u;
#pragma unroll
    for (int j = 0; j < 32; ++j) hits |= (-__uint_as_float(r[j]) <= T ? 1u : 0u) << j;
    const int real = n_class - col_c;                    // columns of this chunk that are references (the rest is padding)
    if (real < 32) hits &= real <= 0 ? 0u : ((1u << real) - 1u);
    while (hits) {
        const int j = __ffs(hits) - 1;
        hits &= hits - 1u;
        const uint32_t pos = atomicAdd(cnt, 1u);
        if (cols) cols[pos] = (uint32_t)(col_c + j);
    }
}

__device__ __forceinline__ void list_tile(uint32_t taddr, int col0, int n_class, float T, uint32_t *cnt, uint32_t *cols) {
    uint32_t ra[32], rb[32];
    __syncwarp();
    tmem_ld32_issue(taddr, ra);
    tmem_wait_ld();
    tmem_ld32_issue(taddr + 32u, rb);
    list_chunk(ra, col0, n_class, T, cnt, cols);
    __syncwarp();
    tmem_wait_ld();
    tmem_ld32_issue(taddr + 64u, ra);
    list_chunk(rb, col0 + 32, n_class, T, cnt, cols);
    __syncwarp();
    tmem_wait_ld();
    tmem_ld32_issue(taddr + 96u, rb);
    list_chunk(ra, col0 + 64, n_class, T, cnt, cols);
    __syncwarp();
    tmem_wait_ld();
    list_chunk(rb, col0 + 96, n_class, T, cnt, cols);
}

struct TcParams {
    int64_t n_points;
    int n_mtiles;
    int nt_ref, nt_pos, nt_neg;          // column tiles of each class (each class padded to a multiple of 128 rows)
    int n_refs, n_cent_pos, n_cent_neg;  // real columns of each class
    const __half *b_img;                 // reference operand, one 16 KB shared-memory image per (tile, K chunk)
    const __half *bx_img;                // extra K columns of the references, one 4 KB no-swizzle image per tile
    const __half *ax_img;                // extra K columns of the query rows, one 4 KB no-swizzle image per 128 rows
    const float *nbs;                    // [(nt_ref + nt_pos + nt_neg) * 128] 2^23 |b'|^2, PAD_NORM on padding rows
    const float *pnorm;                  // same layout: P_j = |B~_j| rounded up, 0 on padding rows
    const float *crow;                   // [n_points] C_row (NaN for a NaN feature row)
    const PrepConsts *consts;            // rho and pmax of the reference set (device)
    uint2 *cand;                         // [n_points, 16] (lower bound as float bits, column within its class)
    float *cand_up;                      // [n_points, 16] matching upper bounds (lower + 2 C P)
    int ref_pad, cp_pad;                 // offsets of the centroid classes in nbs / pnorm
    int skip_scan;                       // option score_force_fallback: the epilogue keeps nothing
    uint32_t *meta;                      // [n_points] cnt_ref | cnt_pos << 8 | cnt_neg << 16 | flags << 24 (1 = centroid overflow)
    float2 *drop_lo;                     // [n_points] smallest lower bound of a dropped negative (.x) / positive (.y) reference
    float *thr_out;                      // [n_points] the row's final threshold: k-th smallest upper bound over every reference seen, kept or dropped
    // list mode (template flag LIST): map_a / crow describe the compacted rows, n_mtiles is derived from *list_count
    const unsigned long long *list_count; int list_max_rows;
    const float *list_thr;               // [list rows] final threshold of the row
    uint32_t *list_cnt;                  // [list rows] references listed so far
    const uint32_t *list_off;            // [list rows] start of the row's range in list_cols (fill pass), LIST_NO_ROOM = skip
    uint32_t *list_cols;                 // pool of listed columns; nullptr = counting pass
};

// Work items of one CTA: contig tiles (first pass) or (contig tile, reference slice) pairs (list pass); every role of the CTA
// walks the same sequence.
struct TcSchedule { int n_items, n_slices; long long n_rows; };
template <bool LIST>
__device__ __forceinline__ TcSchedule tc_schedule(const TcParams &p) {
    TcSchedule s;
    if (!LIST) { s.n_items = p.n_mtiles; s.n_slices = 1; s.n_rows = p.n_points; return s; }
    unsigned long long cnt = *p.list_count;
    if (cnt > (unsigned long long)p.list_max_rows) cnt = (unsigned long long)p.list_max_rows;
    const int n_mt = (int)((cnt + MT - 1) / MT);
    int slices = n_mt ? (int)gridDim.x / n_mt : 1;
    slices = slices < 1 ? 1 : (slices > p.nt_ref ? p.nt_ref : slices);
    s.n_items = n_mt * slices; s.n_slices = slices; s.n_rows = (long long)cnt;
    return s;
}

template <int KN, bool LIST, int NK = NKC>
__global__ void __launch_bounds__(NTHREADS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_a, TcParams p) {
    constexpr bool STREAM = STREAM_A<NK>;
    constexpr int SB = STAGE_BYTES<NK>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t smem_base = smem_u32(smem_raw);
    const uint32_t sm_a = smem_base;                                   // [half 0..1][chunk 0..3] blocks of 16 KB (resident A only)
    const uint32_t sm_b = smem_base + (STREAM ? 0 : A_BYTES);          // NSTAGE stages
    const uint32_t sm_cand = sm_b + NSTAGE * SB;                       // [16 entries][256 rows] x 8 bytes
    const uint32_t sm_stg = sm_cand + CAND_BYTES;                      // [set][nbs | P][128] floats
    const uint32_t sm_x = sm_stg + STG_BYTES;                          // barriers, tmem pointer
    const uint32_t bar_a_full = sm_x + 0, bar_a_empty = sm_x + 8;
    const uint32_t bar_b_full = sm_x + 16, bar_b_empty = sm_x + 16 + 8 * NSTAGE;
    const uint32_t bar_t_full = sm_x + 16 + 16 * NSTAGE, bar_t_empty = bar_t_full + 16;
    const uint32_t bar_n_full = bar_t_empty + 16;                      // nbs / P staging of an accumulator set has landed
    const uint32_t tmem_slot = bar_n_full + 16;
    unsigned char *generic_x = smem_raw + (sm_x - smem_base);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nt_total = p.nt_ref + p.nt_pos + p.nt_neg;

    if (threadIdx.x == 0) {
        if (smem_base & 1023u) __trap();                               // SWIZZLE_128B tiles need 1024-byte alignment
        mbar_init(bar_a_full, 1);
        mbar_init(bar_a_empty, 1);
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(bar_b_full + 8 * s, 1); mbar_init(bar_b_empty + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_t_full + 8 * b, 1);
            mbar_init(bar_t_empty + 8 * b, NEPI / 32);
            mbar_init(bar_n_full + 8 * b, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(generic_x + (tmem_slot - sm_x));
    const TcSchedule sched = tc_schedule<LIST>(p);

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            uint32_t bstage = 0, bphase = 0, tile = 0;
            int it = 0;
            for (int item = blockIdx.x; item < sched.n_items; item += gridDim.x, ++it) {
                const int mt = item / sched.n_slices, sl = item - mt * sched.n_slices;
                const int nt_lo = LIST ? (int)((long long)p.nt_ref * sl / sched.n_slices) : 0;
                const int nt_hi = LIST ? (int)((long long)p.nt_ref * (sl + 1) / sched.n_slices) : nt_total;
                if constexpr (!STREAM) {
                    mbar_wait(bar_a_empty, (uint32_t)((it & 1) ^ 1));
                    mbar_expect_tx(bar_a_full, A_BYTES);
                    for (int h = 0; h < 2; ++h)
                        for (int kc = 0; kc < NKC; ++kc)
                            tma_load_2d(sm_a + (h * NKC + kc) * BLOCK_BYTES, &map_a, bar_a_full, kc * BK, mt * MT + h * BM);
                }
                for (int nt = nt_lo; nt < nt_hi; ++nt, ++tile) {
                    for (int kc = 0; kc < NK; ++kc) {
                        mbar_wait(bar_b_empty + 8 * bstage, bphase ^ 1u);
                        mbar_expect_tx(bar_b_full + 8 * bstage, STREAM ? 3 * BLOCK_BYTES : BLOCK_BYTES);
                        bulk_load(sm_b + bstage * SB, p.b_img + ((int64_t)nt * NK + kc) * (BLOCK_BYTES / 2), BLOCK_BYTES,
                                  bar_b_full + 8 * bstage);
                        if constexpr (STREAM)          // this K-chunk of both A halves travels with the B block (read from L2 per tile)
                            for (int h = 0; h < 2; ++h)
                                tma_load_2d(sm_b + bstage * SB + (1 + h) * BLOCK_BYTES, &map_a, bar_b_full + 8 * bstage, kc * BK, mt * MT + h * BM);
                        if (++bstage == NSTAGE) { bstage = 0; bphase ^= 1u; }
                    }
                    {
                        // fifth slot of the tile: the extra K columns -- the tile's references, then the two row blocks of the contig tile
                        mbar_wait(bar_b_empty + 8 * bstage, bphase ^ 1u);
                        mbar_expect_tx(bar_b_full + 8 * bstage, 3 * XBLK_BYTES);
                        const uint32_t slot = sm_b + bstage * SB;
                        bulk_load(slot, p.bx_img + (int64_t)nt * XBLK_HALVES, XBLK_BYTES, bar_b_full + 8 * bstage);
                        bulk_load(slot + XBLK_BYTES, p.ax_img + (int64_t)(2 * mt) * XBLK_HALVES, 2 * XBLK_BYTES, bar_b_full + 8 * bstage);
                        if (++bstage == NSTAGE) { bstage = 0; bphase ^= 1u; }
                    }
                    // P of this tile for the epilogue's hits, once the epilogue has let go of the set (two tiles ago)
                    const uint32_t set = tile & 1u;
                    mbar_wait(bar_t_empty + 8 * set, ((tile >> 1) & 1u) ^ 1u);
                    mbar_expect_tx(bar_n_full + 8 * set, BN * 4);
                    bulk_load(sm_stg + set * (2 * BN * 4) + BN * 4, p.pnorm + (int64_t)nt * BN, BN * 4, bar_n_full + 8 * set);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        // The whole warp walks the loop so that descriptors and barrier addresses live in uniform registers; one elected
        // lane issues the tensor-core instructions.  Descriptors differ only in their 14-bit address field (16-byte units).
        const uint64_t desc_hi = smem_desc(0) & 0xFFFFFFFF00000000ull;
        const uint32_t desc_lo = (uint32_t)smem_desc(0);
        const uint32_t a_lo = desc_lo | ((sm_a & 0x3FFFFu) >> 4), b_lo = desc_lo | ((sm_b & 0x3FFFFu) >> 4);
        uint32_t bstage = 0, bphase = 0, tile = 0;
        int it = 0;
        for (int item = blockIdx.x; item < sched.n_items; item += gridDim.x, ++it) {
            const int sl = item % sched.n_slices;
            const int nt_lo = LIST ? (int)((long long)p.nt_ref * sl / sched.n_slices) : 0;
            const int nt_hi = LIST ? (int)((long long)p.nt_ref * (sl + 1) / sched.n_slices) : nt_total;
            if constexpr (!STREAM) mbar_wait(bar_a_full, (uint32_t)(it & 1));
            for (int nt = nt_lo; nt < nt_hi; ++nt, ++tile) {
                const uint32_t set = tile & 1u;
                mbar_wait(bar_t_empty + 8 * set, ((tile >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + set * (2 * BN);
#pragma unroll
                for (int kc = 0; kc < NK; ++kc) {
                    mbar_wait(bar_b_full + 8 * bstage, bphase);
                    tc_fence_after();
                    const uint32_t b_blk = b_lo + bstage * (SB >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
#pragma unroll
                            for (int ks = 0; ks < BK / 16; ++ks) {   // 16 halves = 32 bytes along K inside the swizzle row
                                const uint32_t a_blk = STREAM ? b_blk + (1 + h) * (BLOCK_BYTES >> 4) + ks * 2
                                                              : a_lo + (h * NKC + kc) * (BLOCK_BYTES >> 4) + ks * 2;
                                umma_f16(tmem_d + h * BN, desc_hi | a_blk, desc_hi | (b_blk + ks * 2), (kc | ks) ? 1u : 0u);
                            }
                        }
                        umma_commit(bar_b_empty + 8 * bstage);    // block reusable once these MMAs have read it
                    }
                    __syncwarp();
                    if (++bstage == NSTAGE) { bstage = 0; bphase ^= 1u; }
                }
                {
                    // the seventeenth k-step: accumulator += (2^10, 2^-1, 2^-12, C16) . (-n1, -n2, -n3, P16)
                    mbar_wait(bar_b_full + 8 * bstage, bphase);
                    tc_fence_after();
                    const uint32_t slot = sm_b + bstage * SB;
                    if (elect_one()) {
                        const uint64_t xb = smem_desc_plain(slot);
#pragma unroll
                        for (int h = 0; h < 2; ++h) umma_f16(tmem_d + h * BN, smem_desc_plain(slot + XBLK_BYTES + h * XBLK_BYTES), xb, 1u);
                        umma_commit(bar_b_empty + 8 * bstage);
                        umma_commit(bar_t_full + 8 * set);            // accumulator set complete
                    }
                    __syncwarp();
                    if (++bstage == NSTAGE) { bstage = 0; bphase ^= 1u; }
                }
            }
            if constexpr (!STREAM) {
                if (elect_one()) umma_commit(bar_a_empty);        // A tile no longer read
                __syncwarp();
            }
        }
    } else {
        // ================= epilogue: 8 warps; thread = contig row = tensor-memory lane =================
        const int q = warp & 3;                                    // tensor-memory lane quarter this warp may read
        const int half = (warp - 2) >> 2;                          // which 128-row MMA block
        const int row_in_tile = half * BM + q * 32 + lane;
        const uint32_t cand_addr = sm_cand + 8u * (uint32_t)row_in_tile;
        uint32_t tile = 0;
        for (int item = blockIdx.x; item < sched.n_items; item += gridDim.x) {
            const int mt = item / sched.n_slices;
            const int64_t row = (int64_t)mt * MT + row_in_tile;
            float C = (row < sched.n_rows) ? c16_up(p.crow[row]) : NAN;   // the value the extra K column carries (rounded up to FP16)
            const bool live = C >= 0.0f;                           // false for padding rows and NaN feature rows
            const float init = live ? INFINITY : -INFINITY;        // -inf: nothing ever qualifies
            if (!live) C = 0.0f;
            if constexpr (LIST) {
                const int sl = item - mt * sched.n_slices;
                const int nt_lo = (int)((long long)p.nt_ref * sl / sched.n_slices), nt_hi = (int)((long long)p.nt_ref * (sl + 1) / sched.n_slices);
                float T = live ? p.list_thr[row] : -INFINITY;
                uint32_t *my_cnt = p.list_cnt + (live ? row : 0);
                uint32_t *my_cols = nullptr;
                if (p.list_cols && live) {
                    const uint32_t off = p.list_off[row];
                    if (off == LIST_NO_ROOM) T = -INFINITY;
                    else my_cols = p.list_cols + off;
                }
                for (int nt = nt_lo; nt < nt_hi; ++nt, ++tile) {
                    const uint32_t set = tile & 1u;
                    mbar_wait(bar_t_full + 8 * set, (tile >> 1) & 1u);
                    mbar_wait(bar_n_full + 8 * set, (tile >> 1) & 1u);      // P of the tile (hits only): issued with the MMAs, long there by now
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + set * (2 * BN) + half * BN;
                    list_tile(taddr, nt * BN, p.n_refs, T, my_cnt, my_cols);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_t_empty + 8 * set);
                }
            } else {
            float ur[KN], up[1], un[1];
#pragma unroll
            for (int i = 0; i < KN; ++i) ur[i] = init;
            up[0] = init; un[0] = init;
            int cnt_r = 0, cnt_p = 0, cnt_n = 0;
            uint32_t flags = 0u;                                   // 1 = a centroid buffer overflowed
            float drop_lo[2] = {INFINITY, INFINITY};               // smallest lower bound of a dropped negative / positive reference

            for (int nt = 0; nt < nt_total; ++nt, ++tile) {
                const uint32_t set = tile & 1u;
                const uint32_t stg = sm_stg + set * (2 * BN * 4);
                mbar_wait(bar_n_full + 8 * set, (tile >> 1) & 1u);
                mbar_wait(bar_t_full + 8 * set, (tile >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + set * (2 * BN) + half * BN;
                if (p.skip_scan) {
                } else if (nt == 0)
                    scan_tile<KN, CAP_R, true, true>(taddr, stg + BN * 4, 0, p.n_refs, C, cand_addr, 0, ur, cnt_r, flags, drop_lo);
                else if (nt < p.nt_ref)
                    scan_tile<KN, CAP_R, false, true>(taddr, stg + BN * 4, nt * BN, p.n_refs, C, cand_addr, 0, ur, cnt_r, flags, drop_lo);
                else if (nt == p.nt_ref)
                    scan_tile<1, CAP_C, true, false>(taddr, stg + BN * 4, 0, p.n_cent_pos, C, cand_addr, CAP_R, up, cnt_p, flags, drop_lo);
                else if (nt < p.nt_ref + p.nt_pos)
                    scan_tile<1, CAP_C, false, false>(taddr, stg + BN * 4, (nt - p.nt_ref) * BN, p.n_cent_pos, C, cand_addr, CAP_R, up, cnt_p, flags, drop_lo);
                else if (nt == p.nt_ref + p.nt_pos)
                    scan_tile<1, CAP_C, true, false>(taddr, stg + BN * 4, 0, p.n_cent_neg, C, cand_addr, CAP_R + CAP_C, un, cnt_n, flags, drop_lo);
                else
                    scan_tile<1, CAP_C, false, false>(taddr, stg + BN * 4, (nt - p.nt_ref - p.nt_pos) * BN, p.n_cent_neg, C, cand_addr, CAP_R + CAP_C, un, cnt_n, flags, drop_lo);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_t_empty + 8 * set);
            }
            // drop what the final thresholds exclude, then publish the row's candidates
            cand_prune<CAP_R>(cand_addr, 0, cnt_r, ur[KN - 1]);
            cand_prune<CAP_C>(cand_addr, CAP_R, cnt_p, up[0]);
            cand_prune<CAP_C>(cand_addr, CAP_R + CAP_C, cnt_n, un[0]);
            if (row < p.n_points) {
                uint2 *out = p.cand + row * NENT;
                float *out_up = p.cand_up + row * NENT;
#pragma unroll
                for (int e = 0; e < NENT; ++e) {
                    const uint2 ent = lds_v2(cand_addr + (uint32_t)e * (NEPI * 8));
                    const bool used = e < CAP_R ? e < cnt_r : (e < CAP_R + CAP_C ? e - CAP_R < cnt_p : e - CAP_R - CAP_C < cnt_n);
                    const int64_t pcol = (int64_t)ent.y + (e < CAP_R ? 0 : (e < CAP_R + CAP_C ? p.ref_pad : p.ref_pad + p.cp_pad));
                    out[e] = ent;
                    // upper bound with the P of that column (all 16 gathers in flight together, once per contig tile)
                    out_up[e] = used ? fmaf(2.0f * C, p.pnorm[pcol], __uint_as_float(ent.x)) : INFINITY;
                }
                p.meta[row] = (uint32_t)cnt_r | ((uint32_t)cnt_p << 8) | ((uint32_t)cnt_n << 16) | (flags << 24);
                p.drop_lo[row] = make_float2(drop_lo[0], drop_lo[1]);
                p.thr_out[row] = ur[KN - 1];
            }
            }   // first pass
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
}

// This lane's features of a W-wide query row (NCH<W> chunk slots, zero beyond W): from the float64 feature matrix, or from raw
// counts divided by the row total (IEEE float64 division, exactly what kmer.normalize_counts does, scripts/kmer.py:219-220).
template <int W>
__device__ __forceinline__ void load_query_row(const double *points, const uint32_t *counts, int64_t row, int lane,
                                               double (&x)[NCH<W>], uint32_t *total_out = nullptr) {
    if (counts) {
        uint32_t c[NCH<W>];
        unsigned long long total = 0;
#pragma unroll
        for (int i = 0; i < NCH<W>; ++i) { c[i] = in_row<W>(lane, i) ? counts[row * W + lane + 32 * i] : 0u; total += c[i]; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(FULL, total, o);
        const double t = (double)total;
        const double r = 1.0 / t;                        // correctly rounded reciprocal, once per row
#pragma unroll
        for (int i = 0; i < NCH<W>; ++i) x[i] = exact_quotient((double)c[i], t, r);
        if (total_out) *total_out = (uint32_t)total;
    } else {
#pragma unroll
        for (int i = 0; i < NCH<W>; ++i) x[i] = in_row<W>(lane, i) ? points[row * W + lane + 32 * i] : 0.0;
    }
}

// ---------------- operand preparation: float64 rows -> centred, 2^12-scaled FP16 + exact residual norms ----------------
// Distances are translation invariant, so every row is shifted by the uniform vector 1/256 before rounding: frequency rows
// sum to 1, which makes |x - u|^2 = |x|^2 - 1/256 about 4.5x smaller than |x|^2 and shrinks every error term with it.
// (Exact distances are always formed from the unshifted float64 rows.)
//
// Reference rows are laid out in a scrambled order, destination row r <- source row (perm_a * r + perm_c) mod n_src with
// perm_a ~ 0.618 n_src coprime to n_src.  The shipped tables are sorted by taxonomy, so distances to a contig run in long
// monotone stretches along the file and the running threshold of the epilogue would be beaten far more often than in an
// exchangeable order; a golden-ratio stride makes every prefix an even sample of the whole file.
// is_ref = 1: reference / centroid rows: FP16 operand, nbs, P, norms, and rho / pmax by atomic max (positive floats order as ints)
// is_ref = 0: query rows: FP16 operand, norms and C_row (reads rho / pmax, so it must run after every is_ref pass)
// W < 256 (canonical features): the row fills the first W operand columns, centred by 1/W; the other columns are written as FP16
// zero and enter none of the sums, so every bound below is the bound of the W-wide vectors.
template <int W>
__global__ void tc_prep_rows_kernel(const double *__restrict__ src, int64_t n_src, int64_t n_rows, int64_t perm_a, int64_t perm_c,
                                    const uint32_t *__restrict__ src_counts, int is_ref, int64_t n_positive, __half *__restrict__ op, double *__restrict__ norm64, double *__restrict__ cnorm64,
                                    float *__restrict__ nbs, float *__restrict__ pnorm, float *__restrict__ crow,
                                    PrepConsts *consts, uint32_t *__restrict__ row_total, __half *__restrict__ bx) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double shift = 1.0 / (double)W;
    float rho = 0.f, pmax = 0.f;
    if (!is_ref) { rho = consts->rho; pmax = consts->pmax; }
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        double s = 0.0, sc = 0.0, sd = 0.0, sh = 0.0;       // |x|^2, |x - u|^2, |B~ - B|^2, |B|^2 (scaled units)
        const int64_t sr = (r < n_src) ? (perm_a * r + perm_c) % n_src : 0;
        double xs[NCH<W>];
        uint32_t total = 0u;
        if (r < n_src) load_query_row<W>(src, src_counts, sr, lane, xs, &total);
        if (row_total && src_counts && lane == 0 && r < n_src) row_total[sr] = total;
#pragma unroll
        for (int i = 0; i < OPW<W> / 32; ++i) {
            const int d = lane + 32 * i;
            // queries: row-major [n, OPW] (fetched by 2-D TMA); references: the shared-memory image of their 128-row tile,
            // [tile][K chunk of 64][row][128 B with the 16-byte pieces XOR-swizzled by row & 7], so that a B block is ONE
            // contiguous 16 KB bulk copy instead of 128 row pieces gathered by a tensor map
            const int64_t o = is_ref ? ((((r >> 7) * NK_OF<W> + (d >> 6)) * BM + (r & 127)) * BK + ((((d >> 3) & 7) ^ (int)(r & 7)) << 3) + (d & 7))
                                     : r * OPW<W> + d;
            if (W == OPW<W> || (i < NCH<W> && in_row<W>(lane, i))) {
                const double x = (r < n_src) ? xs[i < NCH<W> ? i : 0] : shift;
                op[o] = prep_accumulate<W>(x, s, sc, sd, sh);
            } else {
                op[o] = __float2half_rn(0.0f);
            }
        }
        warp_sum4(s, sc, sd, sh, lane);                    // valid in lane 0
        if (lane == 0) {
            const bool real = r < n_src;
            if (norm64 && real) norm64[sr] = s;
            if (cnorm64 && real) cnorm64[sr] = sc;
            const double P = sqrt(sc) * (double)SCALE * (1.0 + 1e-12);     // |B~| (or |A~|), a hair up against the sqrt rounding
            const double dB = sqrt(sd) * (1.0 + 1e-12);
            const double nH = sqrt(sh) * (1.0 + 1e-12);
            if (is_ref) {
                const float nb = real ? (float)(sc * NORM_SCALE) : PAD_NORM;
                nbs[r] = nb;
                // the extra K columns of this reference (see XK): three-way FP16 split of nbs (exact), P rounded UP to FP16
                __half p16 = __float2half_ru(float_up(P));
                __half n1 = __float2half_rn(65504.0f), n2 = n1, n3 = n1;           // padding rows: lower bound +6.7e7, never a hit
                if (real) {
                    n1 = __float2half_rn(nb * (1.0f / 1024.0f));
                    const float r1 = fmaf(-1024.0f, __half2float(n1), nb);         // exact: nb has 24 bits, n1 takes the top 11
                    n2 = __float2half_rn(r1 * 2.0f);
                    const float r2 = fmaf(-0.5f, __half2float(n2), r1);
                    n3 = __float2half_rn(r2 * 4096.0f);
                    const float left = fmaf(-1.0f / 4096.0f, __half2float(n3), r2);
                    // a reference within 1e-6 of the uniform vector would need FP16 subnormals below 2^-24 for its third piece:
                    // give it the widest interval FP16 can carry instead (always a candidate, measured exactly)
                    if (left != 0.0f || __hisinf(n1)) p16 = __float2half_rn(65504.0f);
                } else {
                    p16 = __float2half_rn(0.0f);
                }
                // P as the epilogue uses it for upper bounds: the FP16 value (or a hair more), label (source row < n_positive) in the
                // lowest mantissa bit
                const uint32_t pb = (__float_as_uint(__half2float(p16)) & ~1u) | (uint32_t)(sr < n_positive);
                pnorm[r] = real ? __uint_as_float(pb) : 0.0f;
                {
                    const __half hz = __float2half_rn(0.0f);
                    const __half row16[8] = {__hneg(n1), __hneg(n2), __hneg(n3), p16, hz, hz, hz, hz};
                    uint4 v;
                    memcpy(&v, row16, 16);
                    uint4 *dst = reinterpret_cast<uint4 *>(bx + xrow_offset(r));
                    dst[0] = v;
                    dst[8] = make_uint4(0u, 0u, 0u, 0u);                            // K half 1: 128 bytes further
                }
                if (real && P > 0.0) {
                    atomicMax(reinterpret_cast<int *>(&consts->rho), __float_as_int(float_up((dB + EPS_ACC_OF<NK_OF<W>> * (P + dB)) / P)));
                    atomicMax(reinterpret_cast<int *>(&consts->pmax), __float_as_int(float_up(P)));
                }
            } else if (real) {
                crow[sr] = query_crow(sc, sd, sh, rho, pmax);
            }
        }
    }
}

// ---------------- decision: candidates -> vote / centroid distances, exact float64 where it matters ----------------
struct DecideParams {
    const double *points; const uint32_t *point_counts; int64_t n_points;
    const double *refs; int64_t n_refs; int64_t n_positive;
    int64_t perm_a, perm_c;            // reference candidate index -> original row: (perm_a * idx + perm_c) mod n_refs
    const double *cent_pos; int64_t n_cent_pos;
    const double *cent_neg; int64_t n_cent_neg;
    const double *cnorm_points;        // centred squared norms of the query rows (NaN = NaN feature row)
    const uint32_t *row_total;         // row totals of the count rows (written by whoever prepared the query operands)
    const uint2 *cand; const float *cand_up; const uint32_t *meta; const float2 *drop_lo; const float *thr;
    ScoreOut out;                      // the neighbour report is written by score_decide_kernel<., true> only
    int64_t *fallback_rows; unsigned long long *fallback_count;
    float *stats;                      // when non-null: [0] max |x - exact| / (C P) (must stay <= 1), [1] max |x - exact| in d2 units
    unsigned long long *rows_remeasured;
    // rows with an overflowed buffer but a final threshold: handed to the list pass instead of the exhaustive kernels
    int64_t *list_rows; unsigned long long *list_count; int list_max_rows;
    float *list_thr; double *list_km;
};

// Squared float64 direct-difference distances of a query row (x: this lane's 8 features, lane-strided) to U rows at once.  Every
// exact road measures its (row, reference) and (row, centroid) pairs with this: each lane's fma chain over its features in
// ascending order, then the butterfly xor 16 ... 1, so that the roads agree bit for bit.  U > 1 keeps independent rows in flight
// where a loop over rows is latency-bound.  Rows are W wide; chunk slots beyond W add fma(0, 0, acc) = acc.
template <int W, int U>
__device__ __forceinline__ void warp_d2(const double (&x)[NCH<W>], const double *const (&b)[U], int lane, double (&acc)[U]) {
#pragma unroll
    for (int t = 0; t < U; ++t) acc[t] = 0.0;
#pragma unroll
    for (int i = 0; i < NCH<W>; ++i)
#pragma unroll
        for (int t = 0; t < U; ++t) {
            const double d = in_row<W>(lane, i) ? x[i] - b[t][lane + 32 * i] : 0.0;
            acc[t] = fma(d, d, acc[t]);
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int t = 0; t < U; ++t) acc[t] += __shfl_xor_sync(FULL, acc[t], o);
}
template <int W>
__device__ __forceinline__ double warp_d2(const double (&x)[NCH<W>], const double *b, int lane) {
    const double *const rows[1] = {b};
    double acc[1];
    warp_d2<W>(x, rows, lane, acc);
    return acc[0];
}

__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

// The decision of a row has a SCALAR part -- which of its (at most 16) candidates can still matter, and whether the neighbour vote
// is already settled by the proven intervals -- and a part that needs the whole (W-wide) row: the exact float64 distances to the one
// or two centroids of each class that survive, and to the band of references when the intervals leave the vote open.  Round 1 ran
// everything warp-wide, one row at a time (795 warp instructions per row, issue-bound).  Now a warp takes 32 consecutive rows and
//   A  every LANE settles the scalar part of its own row from the candidate slots (no shuffles, no reductions),
//   B  the WARP walks the rows that need exact distances (all live rows: the centroid term is always exact) with the row's
//      features spread over the lanes; the row total comes from the producer of the counts (histogram kernel or preparation
//      kernel), so the features are formed without a reduction,
//   C  every lane finishes its row: two square roots, a division and a float64 tanh, then coalesced stores.
constexpr uint32_t ROW_DECIDED = 0u, ROW_OPEN = 1u, ROW_FALLBACK = 2u;

__device__ __forceinline__ int64_t cand_ref_index(const DecideParams &p, uint32_t col) {
    return (int64_t)(((unsigned long long)p.perm_a * col + (unsigned long long)p.perm_c) % (unsigned long long)p.n_refs);
}

#ifndef PHM_DECIDE_MIN_CTAS
#define PHM_DECIDE_MIN_CTAS 3
#endif
// NEIGHBORS: the call also reports the k nearest references and the nearest centroid of each class (p.nb).  A row then counts as
// settled only when its k nearest are identified, not merely its vote: every live row re-measures its band (ROW_OPEN), and a row
// with a dropped candidate within reach goes to the overflow road even when its vote is unanimous.  The scores do not change.
// 5-mer rows (W > 256): a lane holds NCH<W> = 16 or 32 doubles of the row and as many of the next one, which do not fit the
// register budget of PHM_DECIDE_MIN_CTAS blocks per SM; those instantiations ask for one block, so that nothing spills.
template <int W> constexpr int DECIDE_MIN_CTAS = W > KDIM ? 1 : PHM_DECIDE_MIN_CTAS;
template <bool FROM_COUNTS, bool NEIGHBORS = false, int W = KDIM>
__global__ void __launch_bounds__(256, DECIDE_MIN_CTAS<W>) score_decide_kernel(DecideParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int kn = p.out.k;
    const bool has_cent = p.n_cent_pos > 0 && p.n_cent_neg > 0;
    for (int64_t base = warp * 32; base < p.n_points; base += n_warps * 32) {
        // ---------------- A: lane = row ----------------
        const int64_t my_row = base + lane;
        bool my_live = false;
        uint32_t state = ROW_DECIDED, band = 0u, keep_p = 0u, keep_n = 0u;
        uint32_t first_p = 0u, first_n = 0u;                        // centroid index of the lowest kept slot of each class
        bool all_cent = false;
        double my_knn = NAN;
        float my_thr = 0.f;
        if (my_row < p.n_points) my_live = !isnan(p.cnorm_points[my_row]);
        if (my_live) {
            const uint32_t meta = p.meta[my_row];
            const int cnt_r = meta & 255, cnt_p = (meta >> 8) & 255, cnt_n = (meta >> 16) & 255;
            const uint4 *cq = reinterpret_cast<const uint4 *>(p.cand + my_row * NENT);          // two (lower bits, column) entries per load
            const float4 *uq = reinterpret_cast<const float4 *>(p.cand_up + my_row * NENT);
            my_thr = p.thr[my_row];
            // ---- k nearest references: slots 0 .. cnt_r - 1 ----
            if (cnt_r < kn) {
                // fewer kept candidates than k: the k smallest upper bounds belonged to candidates that were dropped when the buffer
                // was full.  The kernel's own final threshold (over kept AND dropped candidates) is still valid: list pass.
                state = ROW_FALLBACK;
            } else {
                float lower[CAP_R], upper[CAP_R];
                uint32_t col[CAP_R];
#pragma unroll
                for (int h = 0; h < CAP_R / 2; ++h) {
                    const uint4 e = cq[h];
                    lower[2 * h] = __uint_as_float(e.x); col[2 * h] = e.y;
                    lower[2 * h + 1] = __uint_as_float(e.z); col[2 * h + 1] = e.w;
                }
                {
                    const float4 u0 = uq[0], u1 = uq[1];
                    const float2 u2 = *reinterpret_cast<const float2 *>(p.cand_up + my_row * NENT + 8);
                    upper[0] = u0.x; upper[1] = u0.y; upper[2] = u0.z; upper[3] = u0.w;
                    upper[4] = u1.x; upper[5] = u1.y; upper[6] = u1.z; upper[7] = u1.w;
                    upper[8] = u2.x; upper[9] = u2.y;
                }
                // the k-th smallest upper bound (ties: lower slot first); the bounds are floats, every comparison is exact
                float u_k = INFINITY;
#pragma unroll
                for (int s = 0; s < CAP_R; ++s) {
                    int rank = 0;
#pragma unroll
                    for (int t = 0; t < CAP_R; ++t)
                        rank += (t != s && t < cnt_r && (upper[t] < upper[s] || (upper[t] == upper[s] && t < s))) ? 1 : 0;
                    if (s < cnt_r && rank == kn - 1) u_k = upper[s];
                }
                uint32_t pos_mask = 0u;
#pragma unroll
                for (int s = 0; s < CAP_R; ++s) {
                    if (s < cnt_r && lower[s] <= u_k) {
                        band |= 1u << s;
                        if (cand_ref_index(p, col[s]) < p.n_positive) pos_mask |= 1u << s;
                    }
                }
                const int n_band = __popc(band);
                const float2 dropped = p.drop_lo[my_row];                 // smallest lower bound of a dropped negative / positive reference
                const bool lost_neg = dropped.x <= u_k, lost_pos = dropped.y <= u_k;
                if (lost_neg || lost_pos) {
                    // a dropped candidate could still be among the k nearest: only a unanimous vote over kept AND dropped ones
                    // can be read off
                    if (NEIGHBORS) state = ROW_FALLBACK;
                    else if (pos_mask == band && !lost_neg) my_knn = 1.0;
                    else if (pos_mask == 0u && !lost_pos) my_knn = -1.0;
                    else state = ROW_FALLBACK;
                } else if (!NEIGHBORS && (n_band == kn || pos_mask == 0u || pos_mask == band)) {
                    // the k nearest are exactly the band, or every possible member votes the same way
                    const int pos = (pos_mask == band) ? kn : ((pos_mask == 0u) ? 0 : __popc(pos_mask));
                    my_knn = knn_vote(pos, kn);
                } else {
                    state = ROW_OPEN;                                    // exact distances of the band decide (part B)
                }
            }
            // ---- nearest centroid of each class: slots CAP_R .. (positive), CAP_R + CAP_C .. (negative) ----
            if (has_cent) {
                all_cent = (meta >> 24) != 0u || cnt_p < 1 || cnt_n < 1;  // more than CAP_C centroids inside the nearest one's interval
                if (!all_cent) {
                    float lo_c[2 * CAP_C], up_c[2 * CAP_C];
                    const uint4 e0 = cq[CAP_R / 2], e1 = cq[CAP_R / 2 + 1], e2 = cq[CAP_R / 2 + 2];
                    {
                        lo_c[0] = __uint_as_float(e0.x); lo_c[1] = __uint_as_float(e0.z); lo_c[2] = __uint_as_float(e1.x);
                        lo_c[3] = __uint_as_float(e1.z); lo_c[4] = __uint_as_float(e2.x); lo_c[5] = __uint_as_float(e2.z);
                        const float2 a = *reinterpret_cast<const float2 *>(p.cand_up + my_row * NENT + 10);
                        const float4 b = uq[3];
                        up_c[0] = a.x; up_c[1] = a.y; up_c[2] = b.x; up_c[3] = b.y; up_c[4] = b.z; up_c[5] = b.w;
                    }
                    float u_p = INFINITY, u_n = INFINITY;
#pragma unroll
                    for (int s = 0; s < CAP_C; ++s) {
                        if (s < cnt_p) u_p = fminf(u_p, up_c[s]);
                        if (s < cnt_n) u_n = fminf(u_n, up_c[CAP_C + s]);
                    }
                    const uint32_t col_c[2 * CAP_C] = {e0.y, e0.w, e1.y, e1.w, e2.y, e2.w};
#pragma unroll
                    for (int s = CAP_C - 1; s >= 0; --s) {                 // descending: first_* end up with the LOWEST kept slot
                        if (s < cnt_p && lo_c[s] <= u_p) { keep_p |= 1u << s; first_p = col_c[s]; }
                        if (s < cnt_n && lo_c[CAP_C + s] <= u_n) { keep_n |= 1u << s; first_n = col_c[CAP_C + s]; }
                    }
                }
            }
        }
        const uint32_t my_info = state | (band << 2) | (keep_p << 12) | (keep_n << 15) | ((all_cent ? 1u : 0u) << 18);

        // ---------------- B: warp = row, for every live row of the batch ----------------
        double my_e0 = INFINITY, my_e1 = INFINITY;
        int64_t my_c0 = -1, my_c1 = -1;                                 // NEIGHBORS: index of the nearest centroid of each class
        unsigned todo = __ballot_sync(FULL, my_live && (has_cent || state == ROW_OPEN || p.stats != nullptr));
        // the count row (or feature row) of the NEXT row to do is fetched while the current one is worked on: the loop is a chain of
        // dependent memory accesses per row otherwise
        uint32_t c_nxt[FROM_COUNTS ? NCH<W> : 1], t_nxt = 0u;
        double x_nxt[FROM_COUNTS ? 1 : NCH<W>];
        auto fetch = [&](int rr) {
            const int64_t row = base + rr;
            if (FROM_COUNTS) {
#pragma unroll
                for (int i = 0; i < NCH<W>; ++i) c_nxt[FROM_COUNTS ? i : 0] = in_row<W>(lane, i) ? p.point_counts[row * W + lane + 32 * i] : 0u;
                t_nxt = p.row_total[row];
            } else {
#pragma unroll
                for (int i = 0; i < NCH<W>; ++i) x_nxt[FROM_COUNTS ? 0 : i] = in_row<W>(lane, i) ? p.points[row * W + lane + 32 * i] : 0.0;
            }
        };
        if (todo) fetch(__ffs(todo) - 1);
        while (todo) {
            const int rr = __ffs(todo) - 1;
            todo &= todo - 1;
            const int64_t row = base + rr;
            const uint32_t info = __shfl_sync(FULL, my_info, rr);
            const uint32_t cp0 = __shfl_sync(FULL, first_p, rr), cn0 = __shfl_sync(FULL, first_n, rr);
            double x[NCH<W>];
            if (FROM_COUNTS) {
                const double t = (double)t_nxt;
                const double r = 1.0 / t;                                 // correctly rounded reciprocal, once per row
#pragma unroll
                for (int i = 0; i < NCH<W>; ++i) x[i] = exact_quotient((double)c_nxt[FROM_COUNTS ? i : 0], t, r);
            } else {
#pragma unroll
                for (int i = 0; i < NCH<W>; ++i) x[i] = x_nxt[FROM_COUNTS ? 0 : i];
            }
            if (todo) fetch(__ffs(todo) - 1);
            const uint2 *ent = p.cand + row * NENT;                       // warp-uniform reads below: one broadcast each
            if ((info & 3u) == ROW_OPEN) {
                // undecided: exact distances of the band, k smallest (ties: lower reference index first)
                const uint32_t bnd = (info >> 2) & 1023u;
                double my_d2 = INFINITY;
                int64_t my_idx = 0;
                unsigned rest = bnd;
                while (rest) {
                    const int s = __ffs(rest) - 1;
                    rest &= rest - 1;
                    const int64_t idx = cand_ref_index(p, ent[s].y);
                    const double d = warp_d2<W>(x, p.refs + idx * W, lane);
                    if (lane == s) { my_d2 = d; my_idx = idx; }
                }
                int erank = 0;
                rest = bnd;
                while (rest) {
                    const int s = __ffs(rest) - 1;
                    rest &= rest - 1;
                    const double od = __shfl_sync(FULL, my_d2, s);
                    const int64_t oi = __shfl_sync(FULL, my_idx, s);
                    if (s != lane && (od < my_d2 || (od == my_d2 && oi < my_idx))) ++erank;
                }
                const bool in_band = lane < CAP_R && ((bnd >> lane) & 1u);
                const unsigned top = __ballot_sync(FULL, in_band && erank < kn);
                const unsigned posm = __ballot_sync(FULL, in_band && my_idx < p.n_positive);
                const double knn = knn_vote(__popc(top & posm), kn);
                if (lane == rr) my_knn = knn;
                if (NEIGHBORS && in_band && erank < kn) put_neighbor(p.out.nb.ref_index, p.out.nb.ref_distance, row * kn + erank, my_idx, sqrt(my_d2));
                if (p.rows_remeasured && lane == 0) atomicAdd(p.rows_remeasured, 1ull);
            }
            if (p.stats) {                    // diagnostics: how much of the proven interval the true value uses
                const uint32_t meta = p.meta[row];
                const int cnt_r = meta & 255;
                const double na = p.cnorm_points[row];
                float worst_use = 0.f, worst_abs = 0.f;
                for (int s = 0; s < CAP_R && s < cnt_r; ++s) {
                    const uint2 e = ent[s];
                    const double lo_s = (double)__uint_as_float(e.x), w_s = (double)p.cand_up[row * NENT + s] - lo_s;
                    const double d = warp_d2<W>(x, p.refs + cand_ref_index(p, e.y) * W, lane);
                    const double exact = (d - na) * NORM_SCALE;                 // what the ranking value estimates
                    const double err = fabs(lo_s + 0.5 * w_s - exact);
                    worst_abs = fmaxf(worst_abs, (float)(err / NORM_SCALE));
                    if (w_s > 0.0) worst_use = fmaxf(worst_use, (float)(err / (0.5 * w_s)));
                }
                if (lane == 0) {
                    atomicMax(reinterpret_cast<int *>(p.stats), __float_as_int(worst_use));
                    atomicMax(reinterpret_cast<int *>(p.stats + 1), __float_as_int(worst_abs));
                }
            }
            if (has_cent) {
                double e2[2] = {INFINITY, INFINITY};
                int64_t i2[2] = {INT64_MAX, INT64_MAX};                  // NEIGHBORS: argmin, first on ties
                unsigned rest_p = (info >> 12) & 7u, rest_n = (info >> 15) & 7u;
                if ((info >> 18) & 1u) {
                    // every centroid, exactly (rare); ascending index, so a strict '<' keeps the first of a tie
                    rest_p = 0u; rest_n = 0u;
#pragma unroll
                    for (int cls = 0; cls < 2; ++cls) {
                        const double *cent = cls ? p.cent_neg : p.cent_pos;
                        const int64_t n_c = cls ? p.n_cent_neg : p.n_cent_pos;
                        for (int64_t c = 0; c < n_c; c += 2) {
                            const int64_t c1 = c + 1 < n_c ? c + 1 : c;
                            const double a0 = warp_d2<W>(x, cent + c * W, lane), a1 = warp_d2<W>(x, cent + c1 * W, lane);
                            if (NEIGHBORS) {
                                if (a0 < e2[cls]) { e2[cls] = a0; i2[cls] = c; }
                                if (a1 < e2[cls]) { e2[cls] = a1; i2[cls] = c1; }
                            } else {
                                e2[cls] = fmin(e2[cls], fmin(a0, a1));
                            }
                        }
                    }
                }
                bool first_round = true;                                 // the lowest kept slot of each class came along from part A
                while (rest_p | rest_n) {                              // one candidate of each class per round: both rows in flight
                    const int sp = rest_p ? __ffs(rest_p) - 1 : 0, sn = rest_n ? __ffs(rest_n) - 1 : 0;
                    const uint32_t ip = first_round ? cp0 : ent[CAP_R + sp].y, in_ = first_round ? cn0 : ent[CAP_R + CAP_C + sn].y;
                    first_round = false;
                    const double *const b[2] = {p.cent_pos + (int64_t)(rest_p ? ip : 0u) * W, p.cent_neg + (int64_t)(rest_n ? in_ : 0u) * W};
                    double a[2];
                    warp_d2<W>(x, b, lane, a);
                    const double ap = a[0], an = a[1];
                    if (NEIGHBORS) {
                        // kept slots are not in index order: the tie rule compares indices
                        if (rest_p && (ap < e2[0] || (ap == e2[0] && (int64_t)ip < i2[0]))) { e2[0] = ap; i2[0] = ip; }
                        if (rest_n && (an < e2[1] || (an == e2[1] && (int64_t)in_ < i2[1]))) { e2[1] = an; i2[1] = in_; }
                    } else {
                        if (rest_p) e2[0] = fmin(e2[0], ap);
                        if (rest_n) e2[1] = fmin(e2[1], an);
                    }
                    rest_p &= rest_p - 1;
                    rest_n &= rest_n - 1;
                }
                if (lane == rr) { my_e0 = e2[0]; my_e1 = e2[1]; }
                if (NEIGHBORS && lane == rr) { my_c0 = i2[0]; my_c1 = i2[1]; }
            }
        }

        // ---------------- C: lane = row ----------------
        if (my_row < p.n_points) {
            double km = NAN;
            if (my_live && has_cent) km = kmeans_score(sqrt(my_e0), sqrt(my_e1));
            if (my_live && state == ROW_FALLBACK) {
                bool listed = false;
                if (p.list_rows) {
                    const unsigned long long slot = atomicAdd(p.list_count, 1ull);
                    if (slot < (unsigned long long)p.list_max_rows) {
                        p.list_rows[slot] = my_row; p.list_thr[slot] = my_thr; p.list_km[slot] = km;
                        listed = true;
                    }
                }
                if (!listed) {
                    const unsigned long long slot_out = atomicAdd(p.fallback_count, 1ull);
                    p.fallback_rows[slot_out] = my_row;
                }
            } else {
                put_scores(p.out, my_row, my_knn, km);
            }
            if (NEIGHBORS) {
                // the centroid term of every live row is settled here, whichever road its references take
                if (!my_live) {
                    put_nan_row(p.out, my_row);
                } else {
                    put_neighbor(p.out.nb.cent_index, p.out.nb.cent_distance, 2 * my_row, has_cent ? my_c0 : -1, has_cent ? sqrt(my_e0) : NAN);
                    put_neighbor(p.out.nb.cent_index, p.out.nb.cent_distance, 2 * my_row + 1, has_cent ? my_c1 : -1, has_cent ? sqrt(my_e1) : NAN);
                }
            }
        }
    }
}

// ---------------- extra K columns of the query rows: (2^10, 2^-1, 2^-12, C16, 0 ...) per row, from the row's error constant ----------------
__device__ __forceinline__ void write_ax_row(__half *ax, int64_t row, float c) {
    const bool live = c >= 0.0f;                                       // NaN (empty contig) and padding rows: C = 0, the row keeps nothing anyway
    const __half row16[8] = {__float2half_rn(1024.0f), __float2half_rn(0.5f), __float2half_rn(1.0f / 4096.0f),
                             live ? __float2half_ru(c) : __float2half_rn(0.0f),
                             __float2half_rn(0.0f), __float2half_rn(0.0f), __float2half_rn(0.0f), __float2half_rn(0.0f)};
    uint4 v;
    memcpy(&v, row16, 16);
    uint4 *dst = reinterpret_cast<uint4 *>(ax + xrow_offset(row));
    dst[0] = v;
    dst[8] = make_uint4(0u, 0u, 0u, 0u);                               // K half 1
}
__global__ void __launch_bounds__(256) tc_build_ax_kernel(const float *__restrict__ crow, int64_t n, int64_t n_pad, __half *__restrict__ ax) {
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n_pad; row += (int64_t)gridDim.x * blockDim.x)
        write_ax_row(ax, row, row < n ? crow[row] : NAN);
}

// ---------------- list pass: compaction of its rows, and the exact decision over the listed references ----------------
template <int OW>                                                              // operand width (OPW)
__global__ void __launch_bounds__(256) tc_list_gather_kernel(const __half *__restrict__ a_op, const float *__restrict__ crow,
                                                             const int64_t *__restrict__ list_rows, const unsigned long long *list_count,
                                                             int max_rows, __half *__restrict__ a_list, float *__restrict__ crow_list,
                                                             uint32_t *__restrict__ list_cnt, __half *__restrict__ ax_list) {
    constexpr int V = OW * 2 / 16 / 32;                                        // 16-byte pieces of a row per lane
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long cnt = *list_count;
    if (cnt > (unsigned long long)max_rows) cnt = (unsigned long long)max_rows;
    const int64_t padded = (int64_t)((cnt + MT - 1) / MT) * MT;
    for (int64_t slot = warp; slot < padded; slot += n_warps) {
        uint4 v[V];
        float c = NAN;                                                 // padding rows of the last tile are not live
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] = make_uint4(0u, 0u, 0u, 0u);
        if (slot < (int64_t)cnt) {
            const int64_t row = list_rows[slot];
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = reinterpret_cast<const uint4 *>(a_op)[row * (OW * 2 / 16) + lane + 32 * j];
            c = crow[row];
        }
#pragma unroll
        for (int j = 0; j < V; ++j) reinterpret_cast<uint4 *>(a_list)[slot * (OW * 2 / 16) + lane + 32 * j] = v[j];
        if (lane == 0) { crow_list[slot] = c; list_cnt[slot] = 0u; write_ax_row(ax_list, slot, c); }
    }
}

// exclusive prefix sum of the per-row counts -> ranges in the pool; counts are kept in list_n and cleared for the fill pass
__global__ void __launch_bounds__(1024) tc_list_scan_kernel(const unsigned long long *list_count, int max_rows, unsigned long long pool_entries,
                                                            uint32_t *list_cnt, uint32_t *list_n, uint32_t *list_off) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_base;
    unsigned long long cnt = *list_count;
    if (cnt > (unsigned long long)max_rows) cnt = (unsigned long long)max_rows;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0ull;
    __syncthreads();
    for (unsigned long long i0 = 0; i0 < cnt; i0 += 1024) {
        const unsigned long long i = i0 + threadIdx.x;
        const unsigned long long mine = i < cnt ? list_cnt[i] : 0u;
        unsigned long long incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = s_warp[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(FULL, wi, o);
                if (lane >= o) wi += up;
            }
            s_warp[lane] = wi - w;                                     // exclusive over warps
        }
        __syncthreads();
        const unsigned long long start = s_base + s_warp[warp] + incl - mine;
        if (i < cnt) {
            list_n[i] = (uint32_t)mine;
            list_off[i] = (start + mine <= pool_entries) ? (uint32_t)start : LIST_NO_ROOM;    // a row that does not fit takes no room at all
            list_cnt[i] = 0u;
        }
        __syncthreads();
        if (threadIdx.x == 1023) s_base = start + mine;
        __syncthreads();
    }
}

struct ListDecideParams {
    const double *points; const uint32_t *point_counts;
    const double *refs; int64_t n_refs; int64_t n_positive;
    int64_t perm_a, perm_c;
    const int64_t *list_rows; const unsigned long long *list_count; int list_max_rows;
    const uint32_t *list_n; const uint32_t *list_off; const uint32_t *list_cols; const double *list_km;
    ScoreOut out;                          // the reference report only (the centroids were reported by score_decide_kernel)
    int64_t *fallback_rows; unsigned long long *fallback_count;
    unsigned long long *rows_listed;       // statistics: rows settled here
};

constexpr int TC_KMAX = 5;                 // k_neighbors <= 5 on the tensor-core path
constexpr int LD_U = 4;                    // listed references in flight per warp

// The K nearest (distance, index) pairs seen so far, ascending by nearer(); empty entries are (INFINITY, -1).  A branch-free
// insertion network, so the list stays in registers.
template <int K>
struct TopK {
    double d[K];
    int i[K];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int s = 0; s < K; ++s) { d[s] = INFINITY; i[s] = -1; }
    }
    __device__ __forceinline__ void insert(double v, int id) {
#pragma unroll
        for (int s = K - 1; s > 0; --s) {
            const bool shift = nearer(v, id, d[s - 1], i[s - 1]), here = nearer(v, id, d[s], i[s]);
            i[s] = shift ? i[s - 1] : (here ? id : i[s]);
            d[s] = shift ? d[s - 1] : (here ? v : d[s]);
        }
        if (nearer(v, id, d[0], i[0])) { d[0] = v; i[0] = id; }
    }
};

// A row finished from its k nearest references (squared distances d2, ascending by nearer()) and its kmeans score: vote, scores
// and the reference report.
__device__ __forceinline__ void finish_row(const ScoreOut &o, int64_t row, const double *d2, const int *idx, int64_t n_positive, double km) {
    int pos = 0;
#pragma unroll
    for (int t = 0; t < TC_KMAX; ++t) {
        if (t >= o.k) break;
        pos += idx[t] >= 0 && idx[t] < n_positive;
        put_neighbor(o.nb.ref_index, o.nb.ref_distance, row * o.k + t, idx[t], sqrt(d2[t]));
    }
    put_scores(o, row, knn_vote(pos, o.k), km);
}

// One warp per listed row: float64 direct-difference distance (warp_d2) to each listed reference, k smallest by (distance,
// reference index), vote.  The centroid part of the score was settled by score_decide_kernel.
template <int W>
__global__ void __launch_bounds__(256) score_list_decide_kernel(ListDecideParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long cnt = *p.list_count;
    if (cnt > (unsigned long long)p.list_max_rows) cnt = (unsigned long long)p.list_max_rows;
    const int kn = p.out.k;
    for (int64_t slot = warp; slot < (int64_t)cnt; slot += n_warps) {
        const int64_t row = p.list_rows[slot];
        const uint32_t n = p.list_n[slot], off = p.list_off[slot];
        if (off == LIST_NO_ROOM || n < (uint32_t)kn) {                 // no room in the pool: exhaustive kernels (n < kn cannot happen)
            if (lane == 0) p.fallback_rows[atomicAdd(p.fallback_count, 1ull)] = row;
            continue;
        }
        double x[NCH<W>];
        load_query_row<W>(p.points, p.point_counts, row, lane, x);
        TopK<TC_KMAX> top;
        top.clear();
        const uint32_t *cols = p.list_cols + off;
        for (uint32_t c0 = 0; c0 < n; c0 += LD_U) {
            const double *b[LD_U];
            int idx[LD_U];
#pragma unroll
            for (int t = 0; t < LD_U; ++t) {
                const uint32_t c = c0 + t < n ? c0 + t : n - 1;
                idx[t] = (int)((p.perm_a * (int64_t)cols[c] + p.perm_c) % p.n_refs);
                b[t] = p.refs + (int64_t)idx[t] * W;
            }
            double acc[LD_U];
            warp_d2<W>(x, b, lane, acc);
#pragma unroll
            for (int t = 0; t < LD_U; ++t) {
                if (c0 + t >= n) break;
                top.insert(acc[t], idx[t]);
            }
        }
        if (lane == 0) {
            finish_row(p.out, row, top.d, top.i, p.n_positive, p.list_km[slot]);
            atomicAdd(p.rows_listed, 1ull);
        }
    }
}

// ---------------- rows the decision kernel could not settle: exhaustive float64 ----------------
// Direct-difference float64 distance to EVERY reference and centroid (the same arithmetic score_decide_kernel uses for its
// candidates), k smallest by (distance, index).  The rows are few (candidate-buffer overflow with mixed labels: contigs sitting
// inside a dense cloud of near-identical references), so the grid is small and persistent and reads the row count on the
// device.  When there are fewer rows than CTAs each row is cut into up to FB_SLICES column slices handled by different CTAs;
// the last CTA to finish a row (ticket counter) merges the slices.
constexpr int FB_U = 8;                    // reference rows in flight per warp
constexpr int FB_SLICES = 16;
constexpr int FB_GRID = 148 * 4;
constexpr int FB_BLOCKED_MIN = FB_GRID;    // more fallback rows than this: blocked kernel (references streamed once per 32 rows)
struct FallbackPart { TopK<TC_KMAX> top; double cp, cn; };
struct FallbackParams {
    const double *points; const uint32_t *point_counts;
    const double *refs; int64_t n_refs; int64_t n_positive;
    const double *cent_pos; int64_t n_cent_pos;
    const double *cent_neg; int64_t n_cent_neg;
    const int64_t *rows; const unsigned long long *count;
    FallbackPart *parts;                   // [FB_GRID][FB_SLICES], used only while rows < CTAs
    unsigned int *tickets;                 // [FB_GRID], zero on entry, left zero on exit
    ScoreOut out;                          // the reference report only (the centroids were reported by score_decide_kernel)
};

// kmeans score from the squared distances to the nearest centroid of each class (NaN without both classes)
__device__ __forceinline__ double fallback_km(const FallbackParams &f, double cp, double cn) {
    return (f.n_cent_pos > 0 && f.n_cent_neg > 0) ? kmeans_score(sqrt(cp), sqrt(cn)) : NAN;
}

// k-way merge of `n_lists` (<= FB_SLICES) lists sorted by nearer() -- a list ends at its first empty entry -- into one, with the
// smallest centroid distances of all
__device__ __forceinline__ FallbackPart merge_parts(const FallbackPart *lists, int n_lists) {
    FallbackPart m;
    int head[FB_SLICES];
    for (int w = 0; w < n_lists; ++w) head[w] = 0;
    for (int t = 0; t < TC_KMAX; ++t) {
        int best = -1;
        for (int w = 0; w < n_lists; ++w) {
            if (head[w] >= TC_KMAX || lists[w].top.i[head[w]] < 0) continue;
            if (best < 0 || nearer(lists[w].top.d[head[w]], lists[w].top.i[head[w]], lists[best].top.d[head[best]], lists[best].top.i[head[best]]))
                best = w;
        }
        m.top.d[t] = best < 0 ? INFINITY : lists[best].top.d[head[best]];
        m.top.i[t] = best < 0 ? -1 : lists[best].top.i[head[best]];
        if (best >= 0) ++head[best];
    }
    m.cp = INFINITY; m.cn = INFINITY;
    for (int w = 0; w < n_lists; ++w) { m.cp = fmin(m.cp, lists[w].cp); m.cn = fmin(m.cn, lists[w].cn); }
    return m;
}

// the vote / score of one row from `n_lists` partial lists (one thread)
__device__ __forceinline__ void fallback_finish(const FallbackParams &f, int64_t row, const FallbackPart *lists, int n_lists) {
    const FallbackPart m = merge_parts(lists, n_lists);
    finish_row(f.out, row, m.top.d, m.top.i, f.n_positive, fallback_km(f, m.cp, m.cn));
}

template <int W>
__global__ void __launch_bounds__(256) score_fallback_kernel(FallbackParams f) {
    __shared__ FallbackPart s_part[8];
    __shared__ FallbackPart s_all[FB_SLICES];
    __shared__ unsigned int s_ticket;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long count = *f.count;
    if (count == 0 || count > FB_BLOCKED_MIN) return;          // many rows: score_fallback_blocked_kernel takes them
    int slices = (int)((unsigned long long)gridDim.x / count);
    slices = slices < 1 ? 1 : (slices > FB_SLICES ? FB_SLICES : slices);
    const unsigned long long items = count * (unsigned long long)slices;
    for (unsigned long long it = blockIdx.x; it < items; it += gridDim.x) {
        const unsigned long long ridx = it / slices;
        const int slice = (int)(it % slices);
        const int64_t row = f.rows[ridx];
        const int64_t c_lo = f.n_refs * slice / slices, c_hi = f.n_refs * (slice + 1) / slices;
        double x[NCH<W>];
        load_query_row<W>(f.points, f.point_counts, row, lane, x);
        TopK<TC_KMAX> top;
        top.clear();
        for (int64_t c0 = c_lo + warp; c0 < c_hi; c0 += 8 * FB_U) {   // ascending index per warp (see nearer)
            const double *b[FB_U];
#pragma unroll
            for (int t = 0; t < FB_U; ++t) {
                const int64_t c = c0 + 8 * t;
                b[t] = f.refs + (c < c_hi ? c : c0) * W;
            }
            double acc[FB_U];
            warp_d2<W>(x, b, lane, acc);                     // FB_U independent rows in flight: this loop is latency-bound
#pragma unroll
            for (int t = 0; t < FB_U; ++t) {
                const int64_t c = c0 + 8 * t;
                if (c >= c_hi) break;
                top.insert(acc[t], (int)c);
            }
        }
        double cp = INFINITY, cn = INFINITY;
        if (slice == 0) {
            for (int64_t c = warp; c < f.n_cent_pos; c += 8) cp = fmin(cp, warp_d2<W>(x, f.cent_pos + c * W, lane));
            for (int64_t c = warp; c < f.n_cent_neg; c += 8) cn = fmin(cn, warp_d2<W>(x, f.cent_neg + c * W, lane));
        }
        __syncthreads();                                        // previous item's merge has finished reading shared memory
        if (lane == 0) { s_part[warp].top = top; s_part[warp].cp = cp; s_part[warp].cn = cn; }
        __syncthreads();
        if (threadIdx.x == 0) {
            if (slices == 1) {
                fallback_finish(f, row, s_part, 8);
            } else {
                // this CTA's slice as one sorted list, published for whichever CTA finishes the row last
                f.parts[ridx * FB_SLICES + slice] = merge_parts(s_part, 8);
                __threadfence();
                s_ticket = atomicAdd(&f.tickets[ridx], 1u);
                if (s_ticket == (unsigned)slices - 1) {
                    __threadfence();
                    // the other CTAs' slices, read past L1 (they were written by other SMs)
                    for (int w = 0; w < slices; ++w) {
                        const FallbackPart *src = f.parts + ridx * FB_SLICES + w;
                        for (int i = 0; i < TC_KMAX; ++i) { s_all[w].top.d[i] = __ldcg(&src->top.d[i]); s_all[w].top.i[i] = __ldcg(&src->top.i[i]); }
                        s_all[w].cp = __ldcg(&src->cp); s_all[w].cn = __ldcg(&src->cn);
                    }
                    fallback_finish(f, row, s_all, slices);
                    f.tickets[ridx] = 0u;                       // ready for the next call
                }
            }
        }
    }
}

// Many fallback rows (an enlarged reference set that is a cloud of near-duplicates): 32 rows per CTA share every reference tile,
// which is staged once in shared memory (transposed, padded: conflict-free for lane = reference), so the references are streamed
// from HBM once per 32 rows instead of once per row.  Reference distances only ORDER the neighbours here; the centroid distances,
// whose values reach the score, use the same warp_d2 as every other path.
// 5-mer rows (W > 256) would need 266 / 534 KB that way: a CTA takes 16 / 8 rows there, and the reference tile is staged 256
// features at a time (the distances are summed in the same order, so they are the same bits).
constexpr int FBB_TR = 32, FBB_PITCH = FBB_TR + 1;
template <int W> constexpr int FBB_QW = W <= KDIM ? 4 : 4 * KDIM / W;          // most rows per warp
template <int W> constexpr int FBB_ROWS = 8 * FBB_QW<W>;                       // rows per CTA
template <int W> constexpr int FBB_DS = W <= KDIM ? W : KDIM;                  // features of the reference tile staged at once
template <int W> constexpr int FBB_SMEM = (FBB_ROWS<W> * W + FBB_DS<W> * FBB_PITCH) * 8 + FBB_ROWS<W> * TC_KMAX * 12 + 64;
template <int W> __host__ __device__ constexpr int fbb_qw(int q) { return q < FBB_QW<W> ? q : FBB_QW<W>; }
static_assert(FBB_SMEM<256> <= 232448 && FBB_SMEM<136> <= 232448 && FBB_SMEM<512> <= 232448 && FBB_SMEM<1024> <= 232448,
              "shared memory budget of one sm_100 CTA (blocked fallback)");

template <int W, int QW>                                                   // row width, rows per warp
__device__ __forceinline__ void fallback_block(const FallbackParams &f, unsigned long long blk, unsigned long long count,
                                               double *s_rows, double *s_tile, double *s_d, int *s_i) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kn = f.out.k;
    __syncthreads();
    // this warp's rows into shared memory; their lists start empty
    int64_t my_row[QW];
    double x[QW][NCH<W>];
#pragma unroll
    for (int q = 0; q < QW; ++q) {
        const unsigned long long ridx = blk * (8 * QW) + warp * QW + q;
        my_row[q] = ridx < count ? f.rows[ridx] : -1;
        if (my_row[q] >= 0) load_query_row<W>(f.points, f.point_counts, my_row[q], lane, x[q]);
#pragma unroll
        for (int i = 0; i < NCH<W>; ++i)
            if (in_row<W>(lane, i)) s_rows[(warp * QW + q) * W + lane + 32 * i] = my_row[q] >= 0 ? x[q][i] : 0.0;
        if (lane < TC_KMAX) { s_d[(warp * QW + q) * TC_KMAX + lane] = INFINITY; s_i[(warp * QW + q) * TC_KMAX + lane] = -1; }
    }
    double thr[QW];
#pragma unroll
    for (int q = 0; q < QW; ++q) thr[q] = INFINITY;
    constexpr int DS = FBB_DS<W>;
    for (int64_t c0 = 0; c0 < f.n_refs; c0 += FBB_TR) {
        double acc[QW];
#pragma unroll
        for (int q = 0; q < QW; ++q) acc[q] = 0.0;
        for (int d0 = 0; d0 < W; d0 += DS) {                               // one slice unless W > 256
            __syncthreads();                                               // previous tile (slice) fully consumed
            for (int idx = threadIdx.x; idx < FBB_TR * DS; idx += 256) {
                const int r = (DS == KDIM) ? idx >> 8 : idx / DS, d = (DS == KDIM) ? idx & 255 : idx % DS;
                s_tile[d * FBB_PITCH + r] = (c0 + r < f.n_refs) ? f.refs[(c0 + r) * W + d0 + d] : 0.0;
            }
            __syncthreads();
            const double *xr = s_rows + warp * QW * W + d0;
#pragma unroll 4
            for (int d = 0; d < DS; d += 2) {
                const double b0 = s_tile[d * FBB_PITCH + lane], b1 = s_tile[(d + 1) * FBB_PITCH + lane];
#pragma unroll
                for (int q = 0; q < QW; ++q) {
                    const double2 xx = *reinterpret_cast<const double2 *>(xr + q * W + d);
                    const double t0 = xx.x - b0, t1 = xx.y - b1;
                    acc[q] = fma(t0, t0, acc[q]);
                    acc[q] = fma(t1, t1, acc[q]);
                }
            }
        }
        const bool real = c0 + lane < f.n_refs;
#pragma unroll
        for (int q = 0; q < QW; ++q) {
            unsigned hit = __ballot_sync(FULL, real && acc[q] < thr[q]);
            while (hit) {                                                  // ascending lane = ascending reference index
                const int src = __ffs(hit) - 1;
                hit &= hit - 1;
                const double d = __shfl_sync(FULL, acc[q], src);
                double *ld = s_d + (warp * QW + q) * TC_KMAX;
                int *li = s_i + (warp * QW + q) * TC_KMAX;
                if (lane == 0) list_insert(ld, li, kn, d, (int)(c0 + src));
                __syncwarp();
                thr[q] = ld[kn - 1];
            }
        }
    }
    // centroids (values reach the score: same arithmetic as everywhere else), then the votes
#pragma unroll
    for (int q = 0; q < QW; ++q) {
        if (my_row[q] < 0) continue;
        double cp = INFINITY, cn = INFINITY;
        for (int64_t c = 0; c < f.n_cent_pos; ++c) cp = fmin(cp, warp_d2<W>(x[q], f.cent_pos + c * W, lane));
        for (int64_t c = 0; c < f.n_cent_neg; ++c) cn = fmin(cn, warp_d2<W>(x[q], f.cent_neg + c * W, lane));
        if (lane == 0) {
            const int at = (warp * QW + q) * TC_KMAX;
            finish_row(f.out, my_row[q], s_d + at, s_i + at, f.n_positive, fallback_km(f, cp, cn));
        }
    }
}

template <int W>
__global__ void __launch_bounds__(256) score_fallback_blocked_kernel(FallbackParams f) {
    extern __shared__ __align__(16) unsigned char fbb_raw[];
    double *s_rows = reinterpret_cast<double *>(fbb_raw);                     // [FBB_ROWS][W]
    double *s_tile = s_rows + FBB_ROWS<W> * W;                                // [FBB_DS][33]
    double *s_d = s_tile + FBB_DS<W> * FBB_PITCH;                             // [FBB_ROWS][TC_KMAX]
    int *s_i = reinterpret_cast<int *>(s_d + FBB_ROWS<W> * TC_KMAX);          // [FBB_ROWS][TC_KMAX]
    const unsigned long long count = *f.count;
    if (count <= FB_BLOCKED_MIN) return;
    // rows per warp chosen so that one wave of CTAs covers all rows when it can (the work per CTA is proportional to its rows)
    int qw = (int)((count + (unsigned long long)gridDim.x * 8 - 1) / ((unsigned long long)gridDim.x * 8));
    qw = qw > FBB_QW<W> ? FBB_QW<W> : qw;
    const unsigned long long n_blocks = (count + 8 * qw - 1) / (8 * qw);
    for (unsigned long long blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        switch (qw) {
            case 1: fallback_block<W, 1>(f, blk, count, s_rows, s_tile, s_d, s_i); break;
            case 2: fallback_block<W, fbb_qw<W>(2)>(f, blk, count, s_rows, s_tile, s_d, s_i); break;
            case 3: fallback_block<W, fbb_qw<W>(3)>(f, blk, count, s_rows, s_tile, s_d, s_i); break;
            default: fallback_block<W, fbb_qw<W>(4)>(f, blk, count, s_rows, s_tile, s_d, s_i); break;
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// [rows, opw] FP16 row-major (opw = OPW of the rows: 256, 512 or 1024), box = 64 features x 128 rows, 128-byte swizzle (the UMMA
// K-major canonical layout)
static int make_map(CUtensorMap *map, const void *base, int64_t rows, int opw) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return PHM_E_UNSUPPORTED; }
    cuuint64_t dims[2] = {(cuuint64_t)opw, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)opw * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
    cuuint32_t elem[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, elem,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with %d", (int)r); return PHM_E_CUDA; }
    return PHM_OK;
}

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct TcWorkspace {
    unsigned long long *fallback_count; float *stats; unsigned long long *rows_remeasured; PrepConsts *consts;   // one 512-byte header
    unsigned long long *list_count, *rows_listed;
    int list_max_rows;
    int64_t list_pool_entries;
    int64_t *list_rows; float *list_thr; double *list_km; float *list_crow; uint32_t *list_cnt, *list_n, *list_off, *list_cols; __half *a_list;
    __half *a_op, *b_op;
    __half *ax_img, *bx_img, *ax_list;            // extra K columns (XK per row, no-swizzle 128-row images)
    float *nbs, *pnorm, *crow;
    uint2 *cand; float *cand_up; uint32_t *meta; float2 *drop_lo; float *thr_out;
    double *norm_points, *norm_refs, *norm_cpos, *norm_cneg;
    double *cnorm_points;
    uint32_t *row_total;
    int64_t *fallback_rows;
    FallbackPart *fb_parts; unsigned int *fb_tickets;
    size_t bytes;
};

// operand width of `dim`-wide rows (host side of OPW)
static inline int op_width(int dim) { return dim <= KDIM ? KDIM : dim; }

static TcWorkspace carve_tc(void *ws, int64_t n, int64_t r_pad, int64_t n_refs, int64_t n_cp, int64_t n_cn, int dim) {
    const int opw = op_width(dim);
    TcWorkspace w;
    size_t off = 0;
    unsigned char *base = static_cast<unsigned char *>(ws);
    auto take = [&](size_t bytes) { unsigned char *p = base ? base + off : nullptr; off += align256(bytes); return p; };
    unsigned char *head = take(512);
    w.list_count = reinterpret_cast<unsigned long long *>(head + 256);
    w.rows_listed = reinterpret_cast<unsigned long long *>(head + 320);
    w.fallback_count = reinterpret_cast<unsigned long long *>(head);
    w.stats = reinterpret_cast<float *>(head + 64);
    w.rows_remeasured = reinterpret_cast<unsigned long long *>(head + 128);
    w.consts = reinterpret_cast<PrepConsts *>(head + 192);
    w.a_op = reinterpret_cast<__half *>(take((size_t)n * opw * 2));
    w.b_op = reinterpret_cast<__half *>(take((size_t)r_pad * opw * 2));
    w.bx_img = reinterpret_cast<__half *>(take((size_t)r_pad * XK * 2));
    w.ax_img = reinterpret_cast<__half *>(take((size_t)round_up(n > 0 ? n : 1, MT) * XK * 2));
    w.nbs = reinterpret_cast<float *>(take((size_t)r_pad * 4));
    w.pnorm = reinterpret_cast<float *>(take((size_t)r_pad * 4));
    w.crow = reinterpret_cast<float *>(take((size_t)n * 4));
    w.cand = reinterpret_cast<uint2 *>(take((size_t)n * NENT * 8));
    w.cand_up = reinterpret_cast<float *>(take((size_t)n * NENT * 4));
    w.meta = reinterpret_cast<uint32_t *>(take((size_t)n * 4));
    w.drop_lo = reinterpret_cast<float2 *>(take((size_t)n * 8));
    w.thr_out = reinterpret_cast<float *>(take((size_t)n * 4));
    w.norm_points = reinterpret_cast<double *>(take((size_t)n * 8));
    w.norm_refs = reinterpret_cast<double *>(take((size_t)n_refs * 8));
    w.norm_cpos = reinterpret_cast<double *>(take((size_t)n_cp * 8));
    w.norm_cneg = reinterpret_cast<double *>(take((size_t)n_cn * 8));
    w.cnorm_points = reinterpret_cast<double *>(take((size_t)n * 8));
    w.row_total = reinterpret_cast<uint32_t *>(take((size_t)n * 4));
    w.fallback_rows = reinterpret_cast<int64_t *>(take((size_t)n * 8));
    w.fb_parts = reinterpret_cast<FallbackPart *>(take(sizeof(FallbackPart) * FB_GRID * FB_SLICES));
    w.fb_tickets = reinterpret_cast<unsigned int *>(take(sizeof(unsigned int) * FB_GRID));
    const int64_t lmax = round_up(n, MT) < LIST_MAX_ROWS ? round_up(n, MT) : LIST_MAX_ROWS;
    w.list_max_rows = (int)lmax;
    w.list_rows = reinterpret_cast<int64_t *>(take((size_t)lmax * 8));
    w.list_thr = reinterpret_cast<float *>(take((size_t)lmax * 4));
    w.list_km = reinterpret_cast<double *>(take((size_t)lmax * 8));
    w.list_crow = reinterpret_cast<float *>(take((size_t)lmax * 4));
    w.list_cnt = reinterpret_cast<uint32_t *>(take((size_t)lmax * 4));
    w.list_n = reinterpret_cast<uint32_t *>(take((size_t)lmax * 4));
    w.list_off = reinterpret_cast<uint32_t *>(take((size_t)lmax * 4));
    w.list_pool_entries = lmax * 2048 < LIST_POOL ? lmax * 2048 : LIST_POOL;       // small problems get a small pool (at least 4 M entries)
    if (w.list_pool_entries < ((int64_t)1 << 22)) w.list_pool_entries = (int64_t)1 << 22;
    w.list_cols = reinterpret_cast<uint32_t *>(take((size_t)w.list_pool_entries * 4));
    w.a_list = reinterpret_cast<__half *>(take((size_t)lmax * opw * 2));
    w.ax_list = reinterpret_cast<__half *>(take((size_t)lmax * XK * 2));
    w.bytes = off;
    return w;
}

size_t score_tc_workspace_bytes(int64_t n, int64_t n_refs, int64_t n_cp, int64_t n_cn, int dim) {
    const int64_t r_pad = round_up(n_refs, BN) + round_up(n_cp, BN) + round_up(n_cn, BN);
    return carve_tc(nullptr, n, r_pad, n_refs, n_cp, n_cn, dim).bytes;
}

bool score_tc_supported(int dim, int k_neighbors, int64_t n_refs, int64_t n_cp, int64_t n_cn) {
    return tc_width(dim) && (k_neighbors == 1 || k_neighbors == 3 || k_neighbors == 5) && n_refs >= k_neighbors && n_cp > 0 && n_cn > 0;
}

// rows of `dim` features (one of tc_width)
static int launch_prep(int dim, const double *src, const uint32_t *src_counts, int64_t n_src, int64_t n_rows, int64_t perm_a, int64_t perm_c, int is_ref,
                       int64_t n_positive, __half *op, double *norm64, double *cnorm64, float *nbs, float *pnorm, float *crow, PrepConsts *consts,
                       cudaStream_t st, uint32_t *row_total = nullptr, __half *bx = nullptr) {
    if (n_rows == 0) return PHM_OK;
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    auto kern = dim == CANON_DIM ? tc_prep_rows_kernel<CANON_DIM>
              : dim == KMER5_DIM ? tc_prep_rows_kernel<KMER5_DIM>
              : dim == CANON5_DIM ? tc_prep_rows_kernel<CANON5_DIM> : tc_prep_rows_kernel<KDIM>;
    kern<<<(unsigned)blocks, 256, 0, st>>>(src, n_src, n_rows, perm_a, perm_c, src_counts, is_ref, n_positive, op, norm64, cnorm64, nbs, pnorm,
                                                          crow, consts, row_total, bx);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

static EventRing g_tc_ring;      // brackets of the score_tc_kernel launches (option "time_kernels")
static EventRing g_decide_ring;  // ... and of the score_decide_kernel launches

// score_tc_kernel for k_neighbors k: the first pass (one CTA per contig tile at most; timed for "time_kernels"), or the list pass
// (persistent; the number of rows is read on the device)
template <int NK>
static int launch_tc(bool list, int k, const CUtensorMap &map, const TcParams &p, cudaStream_t st) {
    void (*kern)(CUtensorMap, TcParams);
    switch (k) {
        case 1: kern = list ? score_tc_kernel<1, true, NK> : score_tc_kernel<1, false, NK>; break;
        case 3: kern = list ? score_tc_kernel<3, true, NK> : score_tc_kernel<3, false, NK>; break;
        case 5: kern = list ? score_tc_kernel<5, true, NK> : score_tc_kernel<5, false, NK>; break;
        default: set_error("tensor-core scoring supports k_neighbors 1, 3, 5"); return PHM_E_UNSUPPORTED;
    }
    PHM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES_OF<NK>));
    int grid = sm_count();
    if (!list && grid > p.n_mtiles) grid = p.n_mtiles;
    const bool timed = !list && g_tc_ring.begin(st);
    kern<<<grid, NTHREADS, SMEM_BYTES_OF<NK>, st>>>(map, p);
    PHM_LAUNCH_CHECK();
    if (timed) g_tc_ring.end(st);
    return PHM_OK;
}

int score_tc_last_ms(float *ms) { return g_tc_ring.mean_ms(ms); }
int score_decide_last_ms(float *ms) { return g_decide_ring.mean_ms(ms); }

static void ref_permutation(int64_t n_refs, int64_t *perm_a, int64_t *perm_c) {
    // golden-ratio stride coprime to n_refs (see tc_prep_rows_kernel)
    int64_t pa = (int64_t)(0.6180339887498949 * (double)n_refs);
    if (pa < 1) pa = 1;
    auto gcd = [](int64_t x, int64_t y) { while (y) { const int64_t t = x % y; x = y; y = t; } return x; };
    while (gcd(pa, n_refs) != 1) ++pa;
    *perm_a = pa;
    *perm_c = n_refs / 3;
}

// Reference side of a scoring call: workspace header cleared, references and centroids prepared (they publish rho and pmax).
// `emit` (optional) receives where the query operands belong, for a producer that prepares them itself.
int score_tc_begin(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, QueryEmit *emit) {
    const int64_t n = a.n_points;
    const int64_t ref_pad = round_up(a.n_refs, BN), cp_pad = round_up(a.n_cent_pos, BN), cn_pad = round_up(a.n_cent_neg, BN);
    const int64_t r_pad = ref_pad + cp_pad + cn_pad;
    TcWorkspace w = carve_tc(ws, n, r_pad, a.n_refs, a.n_cent_pos, a.n_cent_neg, a.dim);
    if (ws_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", ws_bytes, w.bytes); return PHM_E_WORKSPACE; }
    PHM_REQUIRE(n < ((int64_t)1 << 31) - MT && r_pad < ((int64_t)1 << 31), "problem too large for 32-bit TMA coordinates");

    PHM_CUDA_CHECK(cudaMemsetAsync(w.fallback_count, 0, 512, st));
    int rc;
    int64_t perm_a, perm_c;
    const int64_t opw = op_width(a.dim);
    ref_permutation(a.n_refs, &perm_a, &perm_c);
    if ((rc = launch_prep(a.dim, a.refs, nullptr, a.n_refs, ref_pad, perm_a, perm_c, 1, a.n_positive, w.b_op, w.norm_refs, nullptr, w.nbs, w.pnorm, nullptr, w.consts, st,
                          nullptr, w.bx_img)) != PHM_OK) return rc;
    if ((rc = launch_prep(a.dim, a.cent_pos, nullptr, a.n_cent_pos, cp_pad, 1, 0, 1, 0, w.b_op + ref_pad * opw, w.norm_cpos, nullptr, w.nbs + ref_pad,
                          w.pnorm + ref_pad, nullptr, w.consts, st, nullptr, w.bx_img + ref_pad * XK)) != PHM_OK) return rc;
    if ((rc = launch_prep(a.dim, a.cent_neg, nullptr, a.n_cent_neg, cn_pad, 1, 0, 1, 0, w.b_op + (ref_pad + cp_pad) * opw, w.norm_cneg, nullptr,
                          w.nbs + ref_pad + cp_pad, w.pnorm + ref_pad + cp_pad, nullptr, w.consts, st, nullptr,
                          w.bx_img + (ref_pad + cp_pad) * XK)) != PHM_OK) return rc;
    if (emit) { emit->op = w.a_op; emit->crow = w.crow; emit->cnorm = w.cnorm_points; emit->total = w.row_total; emit->consts = w.consts; }
    return PHM_OK;
}

int score_tc(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st) {
    int rc = score_tc_begin(a, ws, ws_bytes, st, nullptr);
    if (rc != PHM_OK) return rc;
    return score_tc_finish(a, ws, ws_bytes, st, false);
}

// Query side: operand preparation (unless a producer already filled the QueryEmit buffers), contraction, decision, fallback.
// W: width of the float64 / count rows
template <int W>
static int tc_finish(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, bool queries_prepared) {
    const int64_t n = a.n_points;
    const int64_t ref_pad = round_up(a.n_refs, BN), cp_pad = round_up(a.n_cent_pos, BN), cn_pad = round_up(a.n_cent_neg, BN);
    const int64_t r_pad = ref_pad + cp_pad + cn_pad;
    TcWorkspace w = carve_tc(ws, n, r_pad, a.n_refs, a.n_cent_pos, a.n_cent_neg, W);
    if (ws_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", ws_bytes, w.bytes); return PHM_E_WORKSPACE; }
    int rc;
    int64_t perm_a, perm_c;
    ref_permutation(a.n_refs, &perm_a, &perm_c);
    if (!queries_prepared &&
        (rc = launch_prep(W, a.points, a.point_counts, n, n, 1, 0, 0, 0, w.a_op, w.norm_points, w.cnorm_points, nullptr, nullptr, w.crow, w.consts, st,
                          w.row_total)) != PHM_OK) return rc;

    CUtensorMap map_a;
    if ((rc = make_map(&map_a, w.a_op, n, OPW<W>)) != PHM_OK) return rc;

    TcParams p;
    p.n_points = n;
    p.n_mtiles = (int)((n + MT - 1) / MT);
    p.nt_ref = (int)(ref_pad / BN); p.nt_pos = (int)(cp_pad / BN); p.nt_neg = (int)(cn_pad / BN);
    p.n_refs = (int)a.n_refs; p.n_cent_pos = (int)a.n_cent_pos; p.n_cent_neg = (int)a.n_cent_neg;
    {
        const int64_t n_pad = round_up(n, MT);
        int64_t blocks = (n_pad + 255) / 256;
        if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
        tc_build_ax_kernel<<<(unsigned)blocks, 256, 0, st>>>(w.crow, n, n_pad, w.ax_img);
        PHM_LAUNCH_CHECK();
    }
    p.bx_img = w.bx_img; p.ax_img = w.ax_img;
    p.b_img = w.b_op; p.nbs = w.nbs; p.pnorm = w.pnorm; p.crow = w.crow; p.consts = w.consts; p.cand = w.cand; p.cand_up = w.cand_up; p.meta = w.meta; p.drop_lo = w.drop_lo; p.thr_out = w.thr_out;
    p.ref_pad = (int)ref_pad; p.cp_pad = (int)cp_pad;
    p.skip_scan = score_force_fallback;
    p.list_count = w.list_count; p.list_max_rows = w.list_max_rows; p.list_thr = w.list_thr; p.list_cnt = w.list_cnt;
    p.list_off = w.list_off; p.list_cols = nullptr;
    if ((rc = launch_tc<NK_OF<W>>(false, a.out.k, map_a, p, st)) != PHM_OK) return rc;

    DecideParams r;
    r.points = a.points; r.point_counts = a.point_counts; r.n_points = n;
    r.refs = a.refs; r.n_refs = a.n_refs; r.n_positive = a.n_positive;
    r.perm_a = perm_a; r.perm_c = perm_c;
    r.cent_pos = a.cent_pos; r.n_cent_pos = a.n_cent_pos; r.cent_neg = a.cent_neg; r.n_cent_neg = a.n_cent_neg;
    r.cnorm_points = w.cnorm_points; r.row_total = w.row_total; r.cand = w.cand; r.cand_up = w.cand_up; r.meta = w.meta; r.drop_lo = w.drop_lo; r.thr = w.thr_out;
    r.out = a.out;
    r.fallback_rows = w.fallback_rows; r.fallback_count = w.fallback_count;
    r.stats = score_collect_stats ? w.stats : nullptr;
    r.rows_remeasured = w.rows_remeasured;
    const bool use_list = score_list_pass != 0;
    r.list_rows = use_list ? w.list_rows : nullptr; r.list_count = w.list_count; r.list_max_rows = w.list_max_rows;
    r.list_thr = w.list_thr; r.list_km = w.list_km;
    int64_t blocks = (n + 255) / 256;                                  // a warp takes 32 consecutive rows at a time
    if (blocks > 148 * 16) blocks = 148 * 16;
    const bool timed = g_decide_ring.begin(st);
    const bool nb = a.out.nb.any();
    if (a.point_counts) {
        if (nb) score_decide_kernel<true, true, W><<<(unsigned)blocks, 256, 0, st>>>(r);
        else score_decide_kernel<true, false, W><<<(unsigned)blocks, 256, 0, st>>>(r);
    } else {
        if (nb) score_decide_kernel<false, true, W><<<(unsigned)blocks, 256, 0, st>>>(r);
        else score_decide_kernel<false, false, W><<<(unsigned)blocks, 256, 0, st>>>(r);
    }
    PHM_LAUNCH_CHECK();
    if (timed) g_decide_ring.end(st);

    // rows whose candidate buffer overflowed but whose threshold is final: second tensor-core pass that lists every reference
    // under the threshold, then the exact decision over the lists (row count read on the device: no host synchronisation)
    if (use_list) {
        tc_list_gather_kernel<OPW<W>><<<sm_count(), 256, 0, st>>>(w.a_op, w.crow, w.list_rows, w.list_count, w.list_max_rows, w.a_list, w.list_crow,
                                                                  w.list_cnt, w.ax_list);
        PHM_LAUNCH_CHECK();
        CUtensorMap map_list;
        if ((rc = make_map(&map_list, w.a_list, w.list_max_rows, OPW<W>)) != PHM_OK) return rc;
        TcParams pl = p;
        pl.crow = w.list_crow;
        pl.ax_img = w.ax_list;
        for (int pass = 0; pass < 2; ++pass) {                           // count, prefix sum, fill
            pl.list_cols = pass ? w.list_cols : nullptr;
            if ((rc = launch_tc<NK_OF<W>>(true, a.out.k, map_list, pl, st)) != PHM_OK) return rc;
            if (pass == 0) {
                tc_list_scan_kernel<<<1, 1024, 0, st>>>(w.list_count, w.list_max_rows, (unsigned long long)w.list_pool_entries, w.list_cnt,
                                                        w.list_n, w.list_off);
                PHM_LAUNCH_CHECK();
            }
        }
        ListDecideParams ld;
        ld.points = a.points; ld.point_counts = a.point_counts;
        ld.refs = a.refs; ld.n_refs = a.n_refs; ld.n_positive = a.n_positive;
        ld.perm_a = perm_a; ld.perm_c = perm_c;
        ld.list_rows = w.list_rows; ld.list_count = w.list_count; ld.list_max_rows = w.list_max_rows;
        ld.list_n = w.list_n; ld.list_off = w.list_off; ld.list_cols = w.list_cols; ld.list_km = w.list_km;
        ld.out = a.out;
        ld.fallback_rows = w.fallback_rows; ld.fallback_count = w.fallback_count;
        ld.rows_listed = w.rows_listed;
        score_list_decide_kernel<W><<<sm_count() * 2, 256, 0, st>>>(ld);
        PHM_LAUNCH_CHECK();
    }

    // rows whose candidate buffer overflowed: exhaustive float64, count read on the device
    FallbackParams f;
    f.points = a.points; f.point_counts = a.point_counts;
    f.refs = a.refs; f.n_refs = a.n_refs; f.n_positive = a.n_positive;
    f.cent_pos = a.cent_pos; f.n_cent_pos = a.n_cent_pos; f.cent_neg = a.cent_neg; f.n_cent_neg = a.n_cent_neg;
    f.rows = w.fallback_rows; f.count = w.fallback_count;
    f.out = a.out;
    f.parts = w.fb_parts; f.tickets = w.fb_tickets;
    PHM_CUDA_CHECK(cudaMemsetAsync(w.fb_tickets, 0, sizeof(unsigned int) * FB_GRID, st));
    score_fallback_kernel<W><<<FB_GRID, 256, 0, st>>>(f);              // few rows: column slices across CTAs
    PHM_LAUNCH_CHECK();
    PHM_CUDA_CHECK(cudaFuncSetAttribute(score_fallback_blocked_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, FBB_SMEM<W>));
    score_fallback_blocked_kernel<W><<<sm_count(), 256, FBB_SMEM<W>, st>>>(f);   // many rows: 32 per CTA share the reference stream
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

int score_tc_finish(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, bool queries_prepared) {
    switch (a.dim) {
        case CANON_DIM: return tc_finish<CANON_DIM>(a, ws, ws_bytes, st, queries_prepared);
        case KMER5_DIM: return tc_finish<KMER5_DIM>(a, ws, ws_bytes, st, queries_prepared);
        case CANON5_DIM: return tc_finish<CANON5_DIM>(a, ws, ws_bytes, st, queries_prepared);
        default: return tc_finish<KDIM>(a, ws, ws_bytes, st, queries_prepared);
    }
}

// statistics of the last score_tc call on this workspace
int score_tc_stats(const void *ws, unsigned long long *fallback_rows, float *out3, cudaStream_t st) {
    unsigned char host[512];
    PHM_CUDA_CHECK(cudaMemcpyAsync(host, ws, 512, cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    memcpy(fallback_rows, host, 8);
    memcpy(out3, host + 64, 8);                // [0] bound usage (<= 1 proves the interval), [1] largest ranking error in d2 units
    unsigned long long remeasured = 0;
    memcpy(&remeasured, host + 128, 8);
    out3[2] = (float)remeasured;               // rows whose neighbour vote needed exact re-measurement
    unsigned long long listed = 0;
    memcpy(&listed, host + 320, 8);
    out3[3] = (float)listed;                   // rows settled by the list pass
    return PHM_OK;
}

}  // namespace tc
}  // namespace phm
