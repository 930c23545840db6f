// K1 / K2 / K3: sequence pack, k-mer histogram with fused fold + normalise, and the simple cross-check kernel.
//
// Replaces the interpreted per-base loop of kmer.count_string (reference scripts/kmer.py:42-50) and
// kmer.normalize_counts (scripts/kmer.py:209-221).  See DESIGN.md for the layout and the roofline.
//
// Histogram kernel in one paragraph: persistent warps pull groups of contigs from a global counter.  A warp owns
// a private table of 32-bit counters in shared memory and walks its contig in 512-byte steps (one 128-bit
// streaming load per lane).  Each lane turns its 16 ASCII bases into 32 bits of 2-bit reference codes with a
// handful of SWAR instructions (kmer_swar.h), fetches the 16 bases that follow from its neighbour lane with a
// shuffle, and bumps one counter per window with `red.shared.add`.  For k = 4 the windows are 5-mers taken at
// every SECOND base (a 5-mer holds two consecutive 4-mers), which halves the number of shared-memory atomics;
// the 1024-bin 5-mer table is projected back onto the 256 4-mer bins when the contig is finished.  Chunks that
// hold a non-ATGC byte or a contig boundary take a warp-uniform slow path with an exact per-base blank mask.
#include "score_common.cuh"
#include "kmer_swar.h"

namespace phm {

struct Dec {
    uint32_t s;       // 16 two-bit codes, first base in the top bits
    uint32_t blank;   // both bits of a base set = that base is not a symbol or lies outside the contig
};

// bases [lo, hi) of the chunk belong to the range being counted; `inv` becomes non-zero when the chunk holds a byte that is not a
// symbol (possibly just outside the range: the flag only decides whether the row total needs a reduction)
__device__ __forceinline__ Dec decode_chunk(uint4 raw, int lo, int hi, uint32_t &inv) {
    uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
    Dec d;
    d.s = codes16_be(w);
    d.blank = 0;
    if (any_invalid16(w)) { d.blank = blank_mask16_be(w); inv = 1u; }
    if (lo > 0 || hi < 16) d.blank |= outside_mask16_be(lo, hi);
    return d;
}

template <int K, int STRIDE>
struct HistCfg {
    static constexpr int W = K + STRIDE - 1;             // window width in bases
    static constexpr int TAB_BINS = 1 << (2 * W);
    static constexpr bool PACKED = (K == 5 && STRIDE == 2);   // 6-mer windows in 16-bit counters, two per word (fold6_k5)
    static constexpr int TAB_BYTES = PACKED ? TAB_BINS * 2 : TAB_BINS * 4;
    static constexpr int OUT_BINS = 1 << (2 * K);
    static constexpr int DIRECT_BYTES = (STRIDE > 1) ? OUT_BINS * 4 : 0;
    static constexpr int ALIGN = TAB_BYTES < 16 ? 16 : TAB_BYTES;
    static constexpr int WARP_BYTES = ALIGN + DIRECT_BYTES;
    static constexpr int PRE = (TAB_BYTES >= 16384 || PACKED) ? 5 : 4;   // streaming loads in flight per lane (measured: 2 -> 4 gains 2-3 %, 6 loses occupancy)
    // CTAs of 8 warps the register allocation must leave room for (the small tables are limited by registers, not by shared memory):
    // 5 x 44 KB for the k = 4 stride-2 table (<= 51 registers), 6 for the 4 KB / 1 KB tables (<= 42); the big tables fit 1 or 2 CTAs anyway
    static constexpr int MIN_CTAS = PACKED ? 1 : (STRIDE > 1 ? 5 : (TAB_BYTES <= 4096 ? 6 : 1));
};

// --------------------------------------------------------------------------------------------------
// the histogram kernel
// --------------------------------------------------------------------------------------------------
// EMIT (k = 4, not canonical): the epilogue also writes the tensor-core scorer's query operands for the contig -- FP16 row, error
// constant, centred norm -- so that the scoring stage starts without a preparation pass over the counts (phm_count_score).
// SWZ (canonical output, k >= 5, STRIDE 1): bin y lives at word y ^ (y >> (2K - 5)), i.e. its top five index bits are xor-ed
// into the bank bits.  The reverse-complement gather of the epilogue reads rc(y) for 32 consecutive y at once; rc puts the
// LAST digits of y first, so without the swizzle those 32 reads differ only in their top bits and land in ONE bank (a 32-way
// conflict on every output word, as many shared-memory wavefronts as the whole counting loop); with it both gathers are
// conflict-free.  The canonical look-up table (compact bin -> representative) is staged in shared memory once per CTA and the
// reverse complement is computed arithmetically.
template <int K>
__device__ __forceinline__ uint32_t swz_off(uint32_t off) {            // off = 4 * bin
    constexpr int SH = 2 * K > 5 ? 2 * K - 5 : 0;
    return off ^ ((off >> SH) & 0x7Cu);
}
template <int K>
__device__ __forceinline__ uint32_t revcomp_fast(uint32_t y) {
    uint32_t x = __brev(y) >> (32 - 2 * K);                            // digits reversed, the two bits of each digit swapped
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    return x ^ (0x55555555u & ((1u << (2 * K)) - 1u));                 // A<->T, G<->C: low bit of every digit
}

// --------------------------------------------------------------------------------------------------
// k = 5 as 6-mer windows at every second base, 16-bit counters packed two per word (bin 2w in the low half of word w, bin 2w + 1 in
// the high half): 8 instead of 16 atomics per step and an 8 KB table.  A step adds at most 8 * 32 = 256 to a counter and the table is
// folded at least every FOLD6_STEPS = 248 steps, so no counter and no partial sum of counters passes 63488: the marginal sums are plain
// 32-bit adds on packed halves.  fold6_k5 adds both marginals of the table to the 1024-bin table `direct` and zeroes the 6-mer table.
// Lane l reads words 4l..4l+3 of each of the 16 rows q (128 words per row): bins q*256 + 8l + 2j + h.
//   first 5-mer   x = bin >> 2   = q * 64 + 2l + (j >> 1)          sum over j & 1, h
//   second 5-mer  x = bin & 1023 = (q & 3) * 256 + 8l + 2j + h     sum over q >> 2
// --------------------------------------------------------------------------------------------------
constexpr int FOLD6_STEPS = 248;

__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint2 v) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t hsum16(uint32_t x) { return (x & 0xFFFFu) + (x >> 16); }

__device__ __forceinline__ void fold6_k5(uint32_t tab, uint32_t direct, int lane) {
    __syncwarp();
    uint4 S[4];                          // S[q & 3] = sum over q >> 2 of row q, packed halves
#pragma unroll
    for (int b = 0; b < 4; ++b) S[b] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const uint32_t a = tab + (uint32_t)(q * 512 + lane * 16);
        const uint4 w = lds_v4(a);
        sts_v4_zero(a);                  // only this lane ever reads these 16 bytes during a fold
        S[q & 3].x += w.x; S[q & 3].y += w.y; S[q & 3].z += w.z; S[q & 3].w += w.w;
        const uint32_t d = direct + (uint32_t)(q * 256 + lane * 8);      // first 5-mer: x = q * 64 + 2l, 2l + 1
        uint2 u = lds_v2(d);
        u.x += hsum16(w.x + w.y);
        u.y += hsum16(w.z + w.w);
        sts_v2(d, u);
    }
    __syncwarp();
#pragma unroll
    for (int b = 0; b < 4; ++b) {                                        // second 5-mer: x = b * 256 + 8l .. 8l + 7
        const uint32_t d = direct + (uint32_t)(b * 1024 + lane * 32);
        uint4 u = lds_v4(d), v = lds_v4(d + 16u);
        u.x += S[b].x & 0xFFFFu; u.y += S[b].x >> 16; u.z += S[b].y & 0xFFFFu; u.w += S[b].y >> 16;
        v.x += S[b].z & 0xFFFFu; v.y += S[b].z >> 16; v.z += S[b].w & 0xFFFFu; v.w += S[b].w >> 16;
        sts_v4(d, u); sts_v4(d + 16u, v);
    }
    __syncwarp();
}

// the field's lowest bit lands on bit `lsb` of the result (bits outside the field are not masked)
template <int WW>
__device__ __forceinline__ uint32_t window_raw(uint32_t cur, uint32_t nxt, int p, int lsb) {
    const int sh = 64 - 2 * p - 2 * WW - lsb;
    if (sh >= 32) return cur >> (sh - 32);
    return funnel_r(nxt, cur, (uint32_t)sh);
}
// one 6-mer window into the packed table: word (bin >> 1), half (bin & 1)
__device__ __forceinline__ void post6(uint32_t tab, uint32_t raw1) {       // raw1 = window_raw<6>(.., lsb = 1)
    red_shared_add(tab | (raw1 & 0x1FFCu), (raw1 & 2u) ? 0x10000u : 1u);
}

// --------------------------------------------------------------------------------------------------
// work plan: contigs ordered by length class, very long contigs in tiles
// --------------------------------------------------------------------------------------------------
// Persistent warps draw work items from a global counter.  With contigs drawn in file order, a 100 kb contig drawn near
// the end keeps one warp busy for ~0.2 ms after every other warp has finished, and a genome-size record (kmer.count_directory
// over reference genomes, scripts/kmer.py:143-180) would run on a single warp with the rest of the GPU idle.  So two small
// passes over the offset table (hist_plan_count_kernel, hist_plan_fill_kernel) write a LIST of work items into the caller's
// workspace, ordered by length class -- 64 kb and more, 32 - 64 kb, 16 - 32 kb, shorter; file order inside a class -- and the
// histogram kernel draws from that list, so a launch ends with its shortest items.
//   length >= SPLIT_MIN  the contig is cut into floor(length / TILE) tiles, each an item of the first class.  A tile covers
//                        the windows that START inside it (its range runs K - 1 bases past its end); interior tile boundaries
//                        are multiples of 512 bytes of the sequence buffer, so only the first and the last step of a tile take
//                        the slow path.  Tiles add their folded bins to the contig's output row with global reductions (the row
//                        is zeroed by the planning pass) and hist_finish_kernel turns the finished rows into the requested
//                        outputs (features, scorer operands) afterwards.
// The same two passes plan a span call (phm_kmer_count_spans), with spans instead of records as items (RecordRanges / SpanRanges below).
// An item carries its own range, so the histogram kernel then never reads the offset table.  The plan is switched off ON THE DEVICE
// (item i is contig i, whole, in file order, as in round 1) when no contig reaches SPLIT_MIN -- measured on BASELINE configs[1], 1 M
// contigs of 1 - 100 kb: 4.92 ms with the list against 4.83 ms without; the tail it removes is short because a warp that is alone on
// its SM runs several times faster than one of forty -- or when the list does not fit the workspace.
constexpr int64_t SPLIT_MIN = 131072;
constexpr int64_t TILE = 65536;
constexpr int N_CLASS = 4;
constexpr uint32_t ITEM_TILE = 1u, ITEM_FIRST_TILE = 2u;

struct PlanEntry { int64_t start, end, contig; uint32_t flags, pad; };     // 32 bytes
struct PlanHeader {                                                        // first bytes of the workspace, zeroed per call
    unsigned long long counter;             // work counter of the histogram kernel
    unsigned long long need[N_CLASS];       // list slots every class needs
    unsigned long long filled[N_CLASS];     // ... and has reserved so far
    unsigned long long n_split;             // contigs of SPLIT_MIN bases and more
    unsigned long long first_bad;           // span calls: lowest index of an invalid span (set to ~0 before the count pass)
};
static_assert(sizeof(PlanEntry) == 32 && sizeof(PlanHeader) <= 256, "workspace layout");

__host__ __device__ __forceinline__ uint32_t plan_tiles(int64_t length) {
    return length >= SPLIT_MIN ? (uint32_t)(length / TILE) : 1u;
}
__host__ __device__ __forceinline__ int plan_class(int64_t length) {
    return length >= 65536 ? 0 : (length >= 32768 ? 1 : (length >= 16384 ? 2 : 3));
}

// Where an item's range comes from.  RecordRanges: item c is record c, [off[c], off[c + 1]).  SpanRanges (phm_kmer_count_spans):
// item i is span i = (record, start, end) of an int64[n, 3] array, the range [off[record] + start, off[record] + end); range()
// returns false, with an empty range, for a span that lies outside its record or names no record -- the count pass reports the
// lowest such index and the host stops before the fill pass.  Spans take the list in any case, because no offset table describes
// them: the count pass sets n_split itself and the fill pass never falls back to drawing items in order.
// length() is range()'s end - start (the count pass needs no more); the record forms keep the load order the passes always had.
struct RecordRanges {
    static constexpr bool SPANS = false;
    __device__ __forceinline__ bool range(const int64_t *__restrict__ off, int64_t c, int64_t &start, int64_t &end) const {
        start = off[c]; end = off[c + 1];
        return true;
    }
    __device__ __forceinline__ bool length(const int64_t *__restrict__ off, int64_t c, int64_t &len) const {
        len = off[c + 1] - off[c];
        return true;
    }
};
struct SpanRanges {
    static constexpr bool SPANS = true;
    const int64_t *spans; int64_t n_records;
    __device__ __forceinline__ bool range(const int64_t *__restrict__ off, int64_t i, int64_t &start, int64_t &end) const {
        const int64_t r = spans[3 * i], a = spans[3 * i + 1], b = spans[3 * i + 2];
        start = 0; end = 0;
        if (r < 0 || r >= n_records || a < 0 || b < a) return false;
        const int64_t rs = off[r];
        if (b > off[r + 1] - rs) return false;
        start = rs + a; end = rs + b;
        return true;
    }
    __device__ __forceinline__ bool length(const int64_t *__restrict__ off, int64_t i, int64_t &len) const {
        int64_t start, end;
        const bool ok = range(off, i, start, end);
        len = end - start;
        return ok;
    }
};

template <class Src>
__global__ void __launch_bounds__(256) hist_plan_count_kernel(const int64_t *__restrict__ off, int64_t n, PlanHeader *plan, Src src) {
    __shared__ unsigned long long s_tot[N_CLASS];
    if (threadIdx.x < N_CLASS) s_tot[threadIdx.x] = 0ull;
    __syncthreads();
    unsigned long long mine[N_CLASS] = {0ull, 0ull, 0ull, 0ull};
    uint32_t n_long = 0u;
    int64_t bad = -1;                                                   // this thread's lowest invalid span (indices ascend)
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
        int64_t len;
        if (!src.length(off, c, len) && bad < 0) bad = c;
        const int q = plan_class(len);
        const unsigned long long m = plan_tiles(len);
#pragma unroll
        for (int j = 0; j < N_CLASS; ++j) mine[j] += (q == j) ? m : 0ull;
        if (m > 1ull) n_long = 1u;
    }
    if (Src::SPANS) {
        if (bad >= 0) atomicMin(&plan->first_bad, (unsigned long long)bad);
        if (blockIdx.x == 0 && threadIdx.x == 0) plan->n_split = 1ull;
    } else if (__any_sync(FULL, n_long != 0u) && (threadIdx.x & 31) == 0) {
        atomicAdd(&plan->n_split, 1ull);                                // only "are there any" matters
    }
#pragma unroll
    for (int j = 0; j < N_CLASS; ++j) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mine[j] += __shfl_xor_sync(FULL, mine[j], d);
        if ((threadIdx.x & 31) == 0 && mine[j]) atomicAdd(&s_tot[j], mine[j]);
    }
    __syncthreads();
    if (threadIdx.x < N_CLASS && s_tot[threadIdx.x]) atomicAdd(&plan->need[threadIdx.x], s_tot[threadIdx.x]);
}

// scratch row of a split contig: its counts row, or (when only features are asked for) the first half of its feature row
__device__ __forceinline__ uint32_t *split_row(uint32_t *counts, double *freq, int64_t c, int out_bins) {
    return counts ? counts + c * (int64_t)out_bins : reinterpret_cast<uint32_t *>(freq + c * (int64_t)out_bins);
}

// One block takes 256 consecutive contigs per round: a block-wide exclusive scan of the slots each contig needs, per class, and ONE
// reservation per class and round in the global counters (a reservation per contig would serialise a million atomics on four words).
// Spans: the host has checked that the list fits, after the count pass, before it launches this pass.
template <class Src>
__global__ void __launch_bounds__(256) hist_plan_fill_kernel(const int64_t *__restrict__ off, int64_t n, int k, PlanHeader *plan,
                                                             PlanEntry *entries, unsigned long long cap,
                                                             uint32_t *counts, double *freq, int out_bins, Src src) {
    __shared__ uint32_t s_warp[8][N_CLASS];
    __shared__ unsigned long long s_base[N_CLASS];
    unsigned long long class_base[N_CLASS];
    unsigned long long total = 0;
#pragma unroll
    for (int j = 0; j < N_CLASS; ++j) { class_base[j] = total; total += plan->need[j]; }
    // no plan when the list does not fit, or when no contig needs tiles (the histogram kernel tests the same): measured on 1 M
    // contigs of 1 - 100 kb, drawing them by length class gains less (a lone warp finishes its last contig quickly) than the list costs
    if (!Src::SPANS && (total > cap || plan->n_split == 0ull)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t rounds = (n + 255) / 256;
    for (int64_t r = blockIdx.x; r < rounds; r += gridDim.x) {
        const int64_t c = r * 256 + threadIdx.x;
        int64_t c_end = 0, c_start = 0;
        uint32_t m = 0u;
        int q = 0;
        if (c < n) { src.range(off, c, c_start, c_end); m = plan_tiles(c_end - c_start); q = plan_class(c_end - c_start); }
        uint32_t excl = 0u;
#pragma unroll
        for (int j = 0; j < N_CLASS; ++j) {
            const uint32_t v = (q == j) ? m : 0u;
            uint32_t incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += up;
            }
            if (q == j) excl = incl - v;
            if (lane == 31) s_warp[warp][j] = incl;
        }
        __syncthreads();
        if (threadIdx.x < N_CLASS) {
            uint32_t run = 0u;
            for (int w = 0; w < 8; ++w) { const uint32_t t = s_warp[w][threadIdx.x]; s_warp[w][threadIdx.x] = run; run += t; }
            s_base[threadIdx.x] = run ? atomicAdd(&plan->filled[threadIdx.x], (unsigned long long)run) : 0ull;
        }
        __syncthreads();
        if (c < n) {
            unsigned long long slot = class_base[q] + s_base[q] + s_warp[warp][q] + excl;
            for (uint32_t t = 0; t < m; ++t) {
                PlanEntry e;
                e.start = (t == 0) ? c_start : ((c_start + (int64_t)t * TILE) & ~(int64_t)511);
                e.end = (t + 1 < m) ? (((c_start + (int64_t)(t + 1) * TILE) & ~(int64_t)511) + (k - 1)) : c_end;
                e.contig = c;
                e.flags = (m > 1u) ? (ITEM_TILE | (t == 0 ? ITEM_FIRST_TILE : 0u)) : 0u;
                e.pad = 0u;
                entries[slot + t] = e;
            }
            if (m > 1u) {
                uint32_t *row = split_row(counts, freq, c, out_bins);
                for (int j = 0; j < out_bins; ++j) row[j] = 0u;
            }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void red_global_add(uint32_t *p, uint32_t v) {
    asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// STAGES > 0: the sequence is staged in shared memory by the TMA unit.  Each warp owns STAGES buffers of 512 bytes; lane 0 issues one
// 1-D bulk copy (cp.async.bulk, completing on an mbarrier) per step, STAGES steps ahead, and every lane then reads its 16 bytes
// with one conflict-free 128-bit shared-memory load.  The loads in flight no longer cost registers, so the depth can be whatever
// covers HBM latency with the warps that fit (the big-table kernels, k >= 5, have few).  STAGES = 0: 128-bit streaming loads into
// a register ring.  MEASURED (1 M contigs, option hist_tma): the staged variant is slower -- k = 4: 6.5 vs 5.1 ms, k = 6 canonical
// 16.2 vs 12.6 ms -- the loads were never this kernel's limit and every step now also pays an mbarrier wait, a warp barrier and
// the re-arm; the register ring stays the default.
constexpr int STAGE_BYTES = 512;

// EXPERIMENT, OFF (compile with -DPHM_HIST_DESKEW=1).  The bank of a 5-mer counter is the low five bits of its index: the last 2.5
// bases of the window.  A contig's GC content is anywhere between 25 % and 75 %, so the "G or C" (high) bits of bases 3 and 4 are
// biased and the 32 lanes of an atomic pile up on fewer banks: expected conflict degree 3.9 over the workload against 3.53 for uniform
// banks (simulation and ncu agree).  XOR-ing those two bits with the LOW bits of bases 0 and 1 -- fair coins under Chargaff's second
// rule, and independent of bases 3 and 4 -- makes all five bank bits fair and independent.  Index bit 3 ^= bit 8, bit 1 ^= bit 6 (a
// bijection of the table onto itself); on byte offsets: off ^ ((off >> 5) & 0x28).  The fold reads row y ^ 2 * (y >> 6 & 1) for bin y
// and swaps the word pairs of a row when y's bit 4 is set.  Bit-exact on every test -- and SLOWER: 5.21 against 4.88 ms per 1 M
// contigs.  The two extra instructions per atomic (16 per step) cost more than the 0.4 wavefronts per atomic they save; a per-chunk
// scramble of the stream cannot do it, because windows overlap and a window's index must not depend on bases outside it.
#ifndef PHM_HIST_DESKEW
#define PHM_HIST_DESKEW 0
#endif
__device__ __forceinline__ uint32_t deskew_off(uint32_t off) { return off ^ ((off >> 5) & 0x28u); }

struct HistJob {
    const uint8_t *seq; const int64_t *off; int64_t n_contigs;
    uint32_t *counts; double *freq;
    const uint16_t *rc_lut, *canon_lut; int out_bins;
    PlanHeader *plan; const PlanEntry *entries; unsigned long long cap;      // cap = 0: the planning passes did not run
};

template <int K, int STRIDE, int WARPS, bool EMIT, bool SWZ, int STAGES>
#ifndef PHM_HIST_MIN_CTAS
#define PHM_HIST_MIN_CTAS 5
#endif
__global__ void __launch_bounds__(WARPS * 32, (WARPS == 8 && HistCfg<K, STRIDE>::WARP_BYTES <= 5120) ? PHM_HIST_MIN_CTAS : 1)
kmer_hist_kernel(const __grid_constant__ HistJob job, const __grid_constant__ tc::QueryEmit emit) {
    using Cfg = HistCfg<K, STRIDE>;
    constexpr int W = Cfg::W;
    constexpr bool FUSED = (K == 4 && STRIDE == 2);          // fold and clear of the 5-mer table in one pass
    constexpr bool DESKEW = FUSED && (PHM_HIST_DESKEW != 0); // 5-mer table with de-skewed bank bits (deskew_off)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint8_t *__restrict__ seq = job.seq;
    uint32_t *__restrict__ counts = job.counts;
    double *__restrict__ freq = job.freq;
    const uint16_t *__restrict__ rc_lut = job.rc_lut;
    const uint16_t *__restrict__ canon_lut = job.canon_lut;
    const int out_bins = job.out_bins;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    // tables are aligned to their own size so that (base | offset) is the address of a bin
    const uint32_t base = (smem_u32(smem_raw) + (uint32_t)Cfg::ALIGN - 1u) & ~((uint32_t)Cfg::ALIGN - 1u);
    const uint32_t tab = base + (uint32_t)warp * Cfg::ALIGN;
    const uint32_t direct = base + (uint32_t)WARPS * Cfg::ALIGN + (uint32_t)warp * Cfg::DIRECT_BYTES;
    const uint32_t vst = (STRIDE > 1) ? direct : tab;     // where the folded 4^K histogram is staged
    const bool canonical = rc_lut != nullptr;

    if (Cfg::TAB_BYTES >= 512) {
        for (int i = lane; i < Cfg::TAB_BYTES / 16; i += 32) sts_v4_zero(tab + 16u * i);
    } else {
        for (int i = lane; i < Cfg::TAB_BINS; i += 32) sts_u32(tab + 4u * i, 0u);
    }
    if (STRIDE > 1)
        for (int i = lane; i < Cfg::OUT_BINS / 4; i += 32) sts_v4_zero(direct + 16u * i);
    __syncwarp();
    // canonical look-up table into whichever end of the allocation the alignment left free (one of them has >= ALIGN / 2 bytes)
    uint32_t lut = 0u;
    if (SWZ) {
        const uint32_t raw0 = smem_u32(smem_raw);
        const uint32_t slack = base - raw0;
        const uint32_t tail0 = base + (uint32_t)WARPS * Cfg::WARP_BYTES;
        lut = (slack >= (uint32_t)Cfg::ALIGN - slack) ? raw0 : tail0;
        for (int j = threadIdx.x; j < out_bins; j += WARPS * 32)
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(lut + 2u * j), "h"(canon_lut[j]) : "memory");
        __syncthreads();
    }

    // TMA staging area: after the tables and their alignment slack
    uint32_t stg = 0u, bar = 0u, g_issue = 0u, g_wait = 0u;              // steps issued / consumed by this warp so far (same in every lane)
    if (STAGES > 0) {
        const uint32_t region = smem_u32(smem_raw) + (uint32_t)WARPS * Cfg::WARP_BYTES + (uint32_t)Cfg::ALIGN;
        stg = region + (uint32_t)warp * (STAGES * STAGE_BYTES);
        bar = region + (uint32_t)WARPS * (STAGES * STAGE_BYTES) + (uint32_t)warp * (STAGES * 8);
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) mbar_init(bar + 8u * s, 1u);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }

    // the plan of this call (written by the two planning passes before this launch)
    unsigned long long n_items = (unsigned long long)job.n_contigs;
    bool planned = false;
    if (job.cap > 0) {
        const unsigned long long need = job.plan->need[0] + job.plan->need[1] + job.plan->need[2] + job.plan->need[3];
        if (need <= job.cap && job.plan->n_split != 0ull) { planned = true; n_items = need; }
    }

    // items a warp takes per visit to the work counter: 1 gives the finest balance (5.03 vs 5.10 ms at k = 4); the 16 KB tables
    // of k = 6 prefer 4 (12.5 vs 12.8 ms)
    constexpr int PER_ITEM = (K >= 6) ? 4 : 1;
    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(&job.plan->counter, 1ull);
        item = __shfl_sync(FULL, item, 0) * PER_ITEM;
        if (item >= n_items) break;

        for (int ci = 0; ci < PER_ITEM; ++ci) {
            if (PER_ITEM > 1 && item + ci >= n_items) break;
            int64_t start, end, c;
            bool is_tile = false;
            if (planned) {
                const longlong2 *ep = reinterpret_cast<const longlong2 *>(job.entries + (item + ci));
                const longlong2 e0 = ep[0], e1 = ep[1];
                start = e0.x; end = e0.y; c = e1.x;
                is_tile = ((uint32_t)e1.y & ITEM_TILE) != 0u;
            } else {
                c = (int64_t)(item + ci);
                start = job.off[c]; end = job.off[c + 1];
            }
            uint32_t inv = 0u;                                         // blank bytes met INSIDE the range (not the bytes around it)
            if (end - start >= K) {
                const int64_t c0 = start >> 4;
                const int nchunks = (int)(((end + 15) >> 4) - c0);
                const int startrel = (int)(start - (c0 << 4));
                const int endrel = (int)(end - (c0 << 4));
                const uint4 *gp = reinterpret_cast<const uint4 *>(seq) + c0;
                const int n_iter = (nchunks + 31) >> 5;

                auto load = [&](int it) -> uint4 {
                    const int ch = it * 32 + lane;
                    return (ch < nchunks) ? ldg_stream(gp + ch) : make_uint4(0u, 0u, 0u, 0u);
                };
                // chunks ch_lo .. ch_lo + span - 1 lie wholly inside the range: ONE unsigned comparison tells an edge chunk (or one past
                // the end), and edge chunks and chunks with a byte that is not a symbol share one rare branch
                const int ch_lo = startrel ? 1 : 0;
                const unsigned span = (endrel >> 4) > ch_lo ? (unsigned)((endrel >> 4) - ch_lo) : 0u;
                auto decode = [&](uint4 raw, int it) -> Dec {          // exact blank mask, range boundaries included
                    const int ch = it * 32 + lane;
                    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
                    Dec d;
                    d.s = codes16_be(w);
                    d.blank = 0u;
                    const bool edge = (unsigned)(ch - ch_lo) >= span;
                    if (edge | (any_invalid16(w) != 0u)) {
                        if (ch >= nchunks) return Dec{0u, 0xFFFFFFFFu};
                        if (any_invalid16(w)) { d.blank = blank_mask16_be(w); inv = 1u; }
                        if (edge) d.blank |= outside_mask16_be(startrel - (ch << 4), endrel - (ch << 4));
                    }
                    return d;
                };
                // the windows of one step on the clean path / with per-base blank masks
                auto post_clean = [&](uint32_t cur_s, uint32_t hi_s) {
#pragma unroll
                    for (int p = 0; p < 16; p += STRIDE) {
                        if (Cfg::PACKED) {
                            post6(tab, window_raw<6>(cur_s, hi_s, p, 1));
                        } else {
                            const uint32_t woff = window_offset<W>(cur_s, hi_s, p);
                            red_shared_inc(tab | (SWZ ? swz_off<K>(woff) : (DESKEW ? deskew_off(woff) : woff)));
                        }
                    }
                };
                auto post_masked = [&](const Dec &cur, uint32_t hi_s, uint32_t hi_b) {
#pragma unroll
                    for (int p = 0; p < 16; p += STRIDE) {
                        const uint32_t bl = window_bits<W>(cur.blank, hi_b, p);
                        const uint32_t idx = window_bits<W>(cur.s, hi_s, p);
                        if (bl == 0u) {
                            if (Cfg::PACKED) post6(tab, idx << 1);
                            else red_shared_inc(tab + (SWZ ? swz_off<K>(4u * idx) : (DESKEW ? deskew_off(4u * idx) : 4u * idx)));
                        } else if (STRIDE > 1) {
                            // a partly blank window still holds up to STRIDE clean k-mers
#pragma unroll
                            for (int s = 0; s < STRIDE; ++s) {
                                const int sh = 2 * (W - K - s);
                                const uint32_t kmask = (1u << (2 * K)) - 1u;
                                if (((bl >> sh) & kmask) == 0u) red_shared_inc(direct + 4u * ((idx >> sh) & kmask));
                            }
                        }
                    }
                };

                // PRE 128-bit loads in flight per lane.  The big tables (k >= 5) leave room for few warps per SM, and then the bytes
                // in flight per SM, not the issue rate, decide whether HBM latency is covered.
                constexpr int PRE = (STAGES > 0) ? 2 : Cfg::PRE;
                // TMA path: step `it` = chunks 32 it .. 32 it + 31 of the range, one bulk copy of up to 512 bytes
                auto issue = [&](int it) {
                    const int c_lo = it * 32;
                    int c_n = nchunks - c_lo;
                    if (c_n <= 0) return;
                    c_n = c_n > 32 ? 32 : c_n;
                    const uint32_t s = g_issue % (STAGES > 0 ? STAGES : 1);
                    if (lane == 0) {
                        mbar_expect_tx(bar + 8u * s, (uint32_t)c_n * 16u);
                        bulk_load(stg + s * STAGE_BYTES, gp + c_lo, (uint32_t)c_n * 16u, bar + 8u * s);
                    }
                    ++g_issue;
                };
                auto fetch = [&](int it) -> uint4 {
                    if (it * 32 >= nchunks) return make_uint4(0u, 0u, 0u, 0u);
                    const uint32_t s = g_wait % (STAGES > 0 ? STAGES : 1);
                    mbar_wait(bar + 8u * s, (g_wait / (STAGES > 0 ? STAGES : 1)) & 1u);
                    ++g_wait;
                    return lds_v4(stg + s * STAGE_BYTES + 16u * (uint32_t)lane);     // lanes past the last chunk read stale bytes: decode() blanks them
                };
                if (STAGES > 0) {
#pragma unroll
                    for (int j = 0; j < STAGES; ++j) issue(j);
                }
                Dec cur = decode(STAGES > 0 ? fetch(0) : load(0), 0);
                uint4 ring[PRE - 1];
                if (STAGES == 0) {
#pragma unroll
                    for (int j = 0; j < PRE - 1; ++j) ring[j] = load(1 + j);
                }
#pragma unroll(PRE - 1)
                for (int it = 0; it < n_iter; ++it) {
                    Dec nxt;
                    if (STAGES > 0) {
                        nxt = decode(fetch(it + 1), it + 1);
                        __syncwarp();                                      // every lane has read (and decoded) the buffer of step `it`
                        issue(it + STAGES);                                // ... which is refilled with the step STAGES ahead
                    } else {
                        nxt = decode(ring[0], it + 1);
#pragma unroll
                        for (int j = 0; j + 1 < PRE - 1; ++j) ring[j] = ring[j + 1];
                        ring[PRE - 2] = load(it + PRE);
                    }
                    // the 16 bases that follow this lane's: the next lane's chunk, and for lane 31 lane 0's chunk of the NEXT step --
                    // one rotating shuffle in which lane 0 offers its next chunk (nobody needs its current one)
                    const uint32_t hi_s = __shfl_sync(FULL, lane == 0 ? nxt.s : cur.s, (lane + 1) & 31);
                    const bool dirty = (cur.blank != 0u) | ((lane == 0) & (nxt.blank != 0u));
                    if (!__any_sync(FULL, dirty)) {
                        post_clean(cur.s, hi_s);
                    } else {
                        const uint32_t hi_b = __shfl_sync(FULL, lane == 0 ? nxt.blank : cur.blank, (lane + 1) & 31);
                        post_masked(cur, hi_s, hi_b);
                    }
                    cur = nxt;
                    if (Cfg::PACKED && (it % FOLD6_STEPS) == FOLD6_STEPS - 1 && it + 1 < n_iter) fold6_k5(tab, direct, lane);
                }
            }
            __syncwarp();

            // ---- fold the window table onto the 4^K bins; row total ----
            unsigned long long total = 0;
            // k = 4 at stride 2: the eight folded bins of a lane stay in registers for the outputs below (only the canonical
            // gather needs them back in shared memory)
            constexpr bool KEEP = (STRIDE > 1) && (Cfg::OUT_BINS / 32 <= 8);
            constexpr int NV = KEEP ? Cfg::OUT_BINS / 32 : 1;
            uint32_t vreg[NV];
            if (Cfg::PACKED) {
                if (end - start >= K) fold6_k5(tab, direct, lane);
                for (int i = lane; i < Cfg::OUT_BINS / 4; i += 32) {
                    const uint4 q = lds_v4(direct + 16u * i);
                    total += (unsigned long long)q.x + q.y + q.z + q.w;
                }
            } else if (FUSED) {
                // One pass over the 5-mer table (word = 4 * first 4-mer + fifth base): the lane reads the rows of its eight bins
                // y = lane + 32 i and clears them.  A row's sum is the number of windows whose FIRST 4-mer is y.  The same eight rows
                // also hold, summed over the top base (i >> 1), every window whose SECOND 4-mer is 4 * (y & 63) + fifth base: the lane
                // owns those eight sums completely, adds them to the table of directly counted 4-mers (two 128-bit read-modify-writes
                // at word 4 * (y & 63)), and after a warp barrier picks up, at y, the second 4-mers and directly counted 4-mers of
                // its own bins.  96 shared-memory wavefronts per contig, fold and clear together, against 113 for separate passes.
                uint4 s2[2];
                s2[0] = make_uint4(0u, 0u, 0u, 0u); s2[1] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    // de-skewed table: bin y = lane + 32 i lives in row y ^ 2 * (bit 6 of y) = (lane ^ 2 * (i >> 1 & 1)) + 32 i
                    const uint32_t a = tab + 16u * (uint32_t)((DESKEW ? (lane ^ (((i >> 1) & 1) << 1)) : lane) + 32 * i);
                    const uint4 q = lds_v4(a);
                    sts_v4_zero(a);
                    vreg[i] = q.x + q.y + q.z + q.w;
                    s2[i & 1].x += q.x; s2[i & 1].y += q.y; s2[i & 1].z += q.z; s2[i & 1].w += q.w;
                }
                if (DESKEW && (lane & 16)) {
                    // ... and the fifth base's high bit is flipped in the rows of bins with bit 4 set (all of this lane's, or none)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint4 t = s2[h];
                        s2[h] = make_uint4(t.z, t.w, t.x, t.y);
                    }
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t a = direct + 16u * (uint32_t)(lane + 32 * h);
                    uint4 d = lds_v4(a);
                    d.x += s2[h].x; d.y += s2[h].y; d.z += s2[h].z; d.w += s2[h].w;
                    sts_v4(a, d);
                }
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    vreg[i] += lds_u32(direct + 4u * (uint32_t)(lane + 32 * i));
                    total += vreg[i];
                }
                __syncwarp();
                sts_v4_zero(direct + 16u * (uint32_t)lane);
                sts_v4_zero(direct + 16u * (uint32_t)(lane + 32));
            } else if (STRIDE > 1) {
#pragma unroll(KEEP ? Cfg::OUT_BINS / 32 : 1)
                for (int i = 0; i < Cfg::OUT_BINS / 32; ++i) {
                    const int y = lane + 32 * i;
                    uint32_t v = lds_u32(direct + 4u * y);
                    const uint4 q = lds_v4(tab + 16u * y);                 // windows whose first k-mer is y
                    v += q.x + q.y + q.z + q.w;
#pragma unroll
                    for (int cc = 0; cc < 4; ++cc) v += lds_u32(tab + 4u * (cc * Cfg::OUT_BINS + y));   // ... whose second k-mer is y
                    if (!KEEP || canonical) sts_u32(direct + 4u * y, v);
                    if (KEEP) vreg[KEEP ? i : 0] = v;
                    total += v;
                }
            } else if (Cfg::OUT_BINS >= 128) {
                for (int i = lane; i < Cfg::OUT_BINS / 4; i += 32) {
                    const uint4 q = lds_v4(tab + 16u * i);
                    total += (unsigned long long)q.x + q.y + q.z + q.w;
                }
            } else {
                for (int y = lane; y < Cfg::OUT_BINS; y += 32) total += lds_u32(tab + 4u * y);
            }
            if (FUSED && canonical) {
                // the canonical gather reads the folded bins from shared memory
#pragma unroll
                for (int i = 0; i < NV; ++i) sts_u32(direct + 4u * (uint32_t)(lane + 32 * i), vreg[i]);
            }
            __syncwarp();

            if (is_tile) {
                // ---- a tile: add the folded bins to the contig's row (hist_finish_kernel derives the other outputs from it) ----
                uint32_t *row = split_row(counts, freq, c, out_bins);
                if (!canonical) {
                    if (KEEP) {
#pragma unroll
                        for (int i = 0; i < NV; ++i)
                            if (vreg[i]) red_global_add(row + lane + 32 * i, vreg[i]);
                    } else {
                        for (int y = lane; y < Cfg::OUT_BINS; y += 32) {
                            const uint32_t v = lds_u32(vst + 4u * y);
                            if (v) red_global_add(row + y, v);
                        }
                    }
                } else {
                    for (int j = lane; j < out_bins; j += 32) {
                        uint32_t y, r, v;
                        if (SWZ) {
                            uint16_t y16;
                            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(y16) : "r"(lut + 2u * j) : "memory");
                            y = y16;
                            r = revcomp_fast<K>(y);
                            v = lds_u32(vst + swz_off<K>(4u * y));
                            if (r != y) v += lds_u32(vst + swz_off<K>(4u * r));
                        } else {
                            y = canon_lut[j];
                            r = rc_lut[y];
                            v = lds_u32(vst + 4u * y);
                            if (r != y) v += lds_u32(vst + 4u * r);
                        }
                        if (v) red_global_add(row + j, v);
                    }
                }
            } else {
                // The row total of a contig without blank bytes is its number of windows: no reduction.
                if (!__any_sync(FULL, inv != 0u)) {
                    total = (end - start >= K) ? (unsigned long long)(end - start - (K - 1)) : 0ull;
                } else {
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(FULL, total, d);
                }
                const double dtotal = (double)total;
                const double rtotal = 1.0 / dtotal;
                if (!canonical) {
                    if (KEEP) {
#pragma unroll
                        for (int i = 0; i < NV; ++i) {
                            const int y = lane + 32 * i;
                            if (counts) counts[c * Cfg::OUT_BINS + y] = vreg[i];
                            if (freq) freq[c * Cfg::OUT_BINS + y] = exact_quotient((double)vreg[i], dtotal, rtotal);
                        }
                    } else {
                        for (int y = lane; y < Cfg::OUT_BINS; y += 32) {
                            const uint32_t v = lds_u32(vst + 4u * y);
                            if (counts) counts[c * Cfg::OUT_BINS + y] = v;
                            if (freq) freq[c * Cfg::OUT_BINS + y] = exact_quotient((double)v, dtotal, rtotal);
                        }
                    }
                    if (EMIT) {
                        // same arithmetic, element order and reduction tree as tc_prep_rows_kernel on (count / total)
                        double s = 0.0, sc = 0.0, sd = 0.0, sh = 0.0;
#pragma unroll
                        for (int i = 0; i < Cfg::OUT_BINS / 32; ++i) {
                            const int y = lane + 32 * i;
                            const double x = exact_quotient((double)(KEEP ? vreg[KEEP ? i : 0] : lds_u32(vst + 4u * y)), dtotal, rtotal);
                            emit.op[c * Cfg::OUT_BINS + y] = tc::prep_accumulate(x, s, sc, sd, sh);
                        }
                        tc::warp_sum3(sc, sd, sh, lane);
                        if (lane == 0) {
                            emit.cnorm[c] = sc;
                            emit.crow[c] = tc::query_crow(sc, sd, sh, emit.consts->rho, emit.consts->pmax);
                            emit.total[c] = (uint32_t)total;
                        }
                    }
                } else {
                    // reverse-complement fold as a gather over the compact output bins: bin j is represented by y = canon_lut[j]
                    // (y <= rc(y)) and collects its partner unless it is its own reverse complement; stores are contiguous in j
#pragma unroll 4
                    for (int j = lane; j < out_bins; j += 32) {
                        uint32_t y, r, v;
                        if (SWZ) {
                            uint16_t y16;
                            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(y16) : "r"(lut + 2u * j) : "memory");
                            y = y16;
                            r = revcomp_fast<K>(y);
                            v = lds_u32(vst + swz_off<K>(4u * y));
                            if (r != y) v += lds_u32(vst + swz_off<K>(4u * r));
                        } else {
                            y = canon_lut[j];
                            r = rc_lut[y];
                            v = lds_u32(vst + 4u * y);
                            if (r != y) v += lds_u32(vst + 4u * r);
                        }
                        const int64_t o = c * (int64_t)out_bins + j;
                        if (counts) counts[o] = v;
                        if (freq) freq[o] = exact_quotient((double)v, dtotal, rtotal);
                    }
                }
            }
            __syncwarp();

            // ---- clear for the next item (the packed table was zeroed by its fold, the fused one while it was read) ----
            if (Cfg::PACKED) {
            } else if (FUSED) {
            } else if (Cfg::TAB_BINS >= 128) {
                for (int i = lane; i < Cfg::TAB_BINS / 4; i += 32) sts_v4_zero(tab + 16u * i);
            } else {
                for (int i = lane; i < Cfg::TAB_BINS; i += 32) sts_u32(tab + 4u * i, 0u);
            }
            if (STRIDE > 1 && (!FUSED || canonical))
                for (int i = lane; i < Cfg::OUT_BINS / 4; i += 32) sts_v4_zero(direct + 16u * i);
            __syncwarp();
        }
    }
}

// Rows of the split contigs, complete once the histogram kernel has finished: the outputs that derive from a whole row.  One warp
// per first-tile entry of the list's first class (the only class that holds tiles).  When only features were asked for, the row was
// accumulated in the first half of its own feature row; features are then written from the LAST bin down, 32 at a time, each group
// read completely before it is written: feature j overwrites counters 2j and 2j + 1, which no lower group still needs.
template <bool EMIT>
__global__ void __launch_bounds__(256) hist_finish_kernel(const __grid_constant__ HistJob job, const __grid_constant__ tc::QueryEmit emit) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned long long need = job.plan->need[0] + job.plan->need[1] + job.plan->need[2] + job.plan->need[3];
    if (job.cap == 0 || need > job.cap || job.plan->n_split == 0ull) return;
    const unsigned long long n0 = job.plan->need[0];
    const int out_bins = job.out_bins;
    for (unsigned long long i = (unsigned long long)blockIdx.x * 8 + wib; i < n0; i += (unsigned long long)gridDim.x * 8) {
        const PlanEntry e = job.entries[i];
        if (!(e.flags & ITEM_FIRST_TILE)) continue;
        const int64_t c = e.contig;
        volatile uint32_t *row = split_row(job.counts, job.freq, c, out_bins);
        unsigned long long total = 0;
        for (int j = lane; j < out_bins; j += 32) total += row[j];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(FULL, total, d);
        const double dt = (double)total, rdt = 1.0 / dt;
        if (EMIT) {
            double s = 0.0, sc = 0.0, sd = 0.0, sh = 0.0;
#pragma unroll
            for (int t = 0; t < tc::PREP_DIM / 32; ++t) {
                const int y = lane + 32 * t;
                const double x = exact_quotient((double)row[y], dt, rdt);
                emit.op[c * tc::PREP_DIM + y] = tc::prep_accumulate(x, s, sc, sd, sh);
            }
            tc::warp_sum3(sc, sd, sh, lane);
            if (lane == 0) {
                emit.cnorm[c] = sc;
                emit.crow[c] = tc::query_crow(sc, sd, sh, emit.consts->rho, emit.consts->pmax);
                emit.total[c] = (uint32_t)total;
            }
        }
        if (job.freq) {
            __syncwarp();
            for (int j0 = ((out_bins - 1) >> 5) << 5; j0 >= 0; j0 -= 32) {
                const int j = j0 + lane;
                uint32_t v = 0u;
                if (j < out_bins) v = row[j];
                __syncwarp();
                if (j < out_bins) job.freq[c * (int64_t)out_bins + j] = exact_quotient((double)v, dt, rdt);
                __syncwarp();
            }
        }
    }
}

// --------------------------------------------------------------------------------------------------
// sliding windows (phm_window_offsets, phm_kmer_count_windows): every window is one work item of the list above
// --------------------------------------------------------------------------------------------------
// A record of length L has one window [0, L) when L <= w, else the windows [j s, j s + w) while j s + w <= L, plus [L - w, L) when
// the last of those ends before L: 1 + ceil((L - w) / s) windows, each exactly w long.  The histogram kernel counts any range into any
// row, so a window call only needs its own planning pass: window_plan_kernel writes one list entry per window of the slice (row =
// index in the slice), in window order, and the unchanged kmer_hist_kernel / hist_finish_kernel take the list from there.
__host__ __device__ __forceinline__ int64_t windows_of(int64_t len, int64_t w, int64_t s) {
    return len <= w ? 1 : 2 + (len - w - 1) / s;                        // 1 + ceil((len - w) / s) without overflow for any s
}

// Prefix sum of the window counts in three passes that need no scratch memory beyond the output: tiles of WO_TILE records scanned
// locally (window_offsets_kernel), the tiles' last entries scanned in place by one block (window_offsets_carry_kernel), then every
// other entry of a tile adds the finished last entry of the tile before it (window_offsets_add_kernel).
constexpr int WO_PER_THREAD = 8;
constexpr int WO_TILE = 256 * WO_PER_THREAD;

__global__ void __launch_bounds__(256) window_offsets_kernel(const int64_t *__restrict__ off, int64_t n, int64_t w, int64_t s,
                                                             int64_t *__restrict__ wo) {
    __shared__ long long s_warp[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * WO_TILE + (int64_t)threadIdx.x * WO_PER_THREAD;
    int64_t cnt[WO_PER_THREAD], mine = 0;
#pragma unroll
    for (int j = 0; j < WO_PER_THREAD; ++j) {
        const int64_t r = r0 + j;
        cnt[j] = r < n ? windows_of(off[r + 1] - off[r], w, s) : 0;
        mine += cnt[j];
    }
    long long incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int64_t run = incl - mine;
    for (int v = 0; v < warp; ++v) run += s_warp[v];
#pragma unroll
    for (int j = 0; j < WO_PER_THREAD; ++j) {
        run += cnt[j];
        if (r0 + j < n) wo[r0 + j + 1] = run;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) wo[0] = 0;
}

__global__ void __launch_bounds__(1024) window_offsets_carry_kernel(int64_t n, int64_t *wo) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t tiles = (n + WO_TILE - 1) / WO_TILE;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int64_t t0 = 0; t0 < tiles; t0 += 1024) {
        const int64_t t = t0 + threadIdx.x;
        const int64_t at = t < tiles ? ((t + 1) * WO_TILE < n ? (t + 1) * WO_TILE : n) : 0;   // entry of the tile's last record
        const long long v = t < tiles ? wo[at] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        long long before = s_carry;
        for (int q = 0; q < warp; ++q) before += s_warp[q];
        if (t < tiles) wo[at] = before + incl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) window_offsets_add_kernel(int64_t n, int64_t *wo) {
    for (int64_t r = (int64_t)WO_TILE + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t tile_end = (r / WO_TILE + 1) * WO_TILE;
        if (r + 1 == tile_end || r + 1 == n) continue;                       // the tile's last entry is already final
        wo[r + 1] += wo[(r / WO_TILE) * WO_TILE];
    }
}

// One thread per window of the slice [first, first + n): its record by binary search in the window offsets, its range, and the list
// entries of its row.  Every window gets `per` slots (the tiles of a w-long window): a window of SPLIT_MIN bases and more is cut by
// the rule of hist_plan_fill_kernel (its row zeroed, first tile flagged for hist_finish_kernel); a shorter one (only the single window
// of a record shorter than w can be) fills its first slot and pads the others with empty tiles, which count nothing and add nothing.
// The header makes the histogram kernel take the list: `need` in the class the host chose (class 0 when windows are tiled, the only
// class hist_finish_kernel walks) and n_split != 0.
__global__ void __launch_bounds__(256) window_plan_kernel(const int64_t *__restrict__ off, const int64_t *__restrict__ wo, int64_t n_records,
                                                          int64_t w, int64_t s, int64_t first, int64_t n, int k, uint32_t per, int cls,
                                                          PlanHeader *plan, PlanEntry *entries, uint32_t *counts, double *freq, int out_bins,
                                                          int64_t *spans) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        plan->need[cls] = (unsigned long long)n * per;
        plan->n_split = 1ull;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t g = first + i;
        int64_t lo = 0, hi = n_records;                                     // wo[lo] <= g < wo[hi]
        while (hi - lo > 1) {
            const int64_t mid = lo + ((hi - lo) >> 1);
            if (wo[mid] <= g) lo = mid; else hi = mid;
        }
        const int64_t rs = off[lo], len = off[lo + 1] - rs, j = g - wo[lo];
        int64_t a = 0, b = len;
        if (len > w) {
            a = (j + 1 < windows_of(len, w, s)) ? j * s : len - w;
            b = a + w;
        }
        if (spans) { spans[2 * i] = a; spans[2 * i + 1] = b; }
        const int64_t c_start = rs + a, c_end = rs + b;
        const uint32_t m = plan_tiles(b - a);
        for (uint32_t t = 0; t < per; ++t) {
            PlanEntry e;
            e.contig = i;
            e.pad = 0u;
            if (t >= m) {
                e.start = c_start; e.end = c_start; e.flags = ITEM_TILE;
            } else if (m == 1u) {
                e.start = c_start; e.end = c_end; e.flags = 0u;
            } else {
                e.start = (t == 0) ? c_start : ((c_start + (int64_t)t * TILE) & ~(int64_t)511);
                e.end = (t + 1 < m) ? (((c_start + (int64_t)(t + 1) * TILE) & ~(int64_t)511) + (k - 1)) : c_end;
                e.flags = ITEM_TILE | (t == 0 ? ITEM_FIRST_TILE : 0u);
            }
            entries[(unsigned long long)i * per + t] = e;
        }
        if (m > 1u) {
            uint32_t *row = split_row(counts, freq, i, out_bins);
            for (int q = 0; q < out_bins; ++q) row[q] = 0u;
        }
    }
}

// --------------------------------------------------------------------------------------------------
// canonical look-up tables: rc[y] and compact[y] = rank of min(y, rc(y)) among the self-representing bins
// --------------------------------------------------------------------------------------------------
__global__ void canonical_lut_kernel(int k, uint16_t *rc_lut, uint16_t *compact_lut, uint16_t *canon_lut) {
    __shared__ uint16_t rank[4096];
    const int bins = 1 << (2 * k);
    for (int y = threadIdx.x; y < bins; y += blockDim.x) rc_lut[y] = (uint16_t)revcomp_bin((uint32_t)y, k);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint16_t r = 0;
        for (int y = 0; y < bins; ++y) {
            rank[y] = r;
            if ((uint32_t)y <= rc_lut[y]) ++r;
        }
    }
    __syncthreads();
    for (int y = threadIdx.x; y < bins; y += blockDim.x) {
        const uint32_t r = rc_lut[y];
        compact_lut[y] = rank[r < (uint32_t)y ? r : y];
        if ((uint32_t)y <= r) canon_lut[rank[y]] = (uint16_t)y;      // compact bin -> its representative
    }
}

// --------------------------------------------------------------------------------------------------
// canonical fold of rows that already exist (phm_canonical_fold): float64 [n, 4^K] -> [n, canonical bins], the counter's definition
// and bin order.  Every CTA builds the compact bin -> representative table in shared memory (a block scan over y <= rc(y)), so the
// call needs no workspace; then a warp per row writes out[c] = row[y] + row[rc(y)] for the representative y of c (row[y] alone
// when y is its own reverse complement): one add per bin pair, exact for integer rows below 2^53.
// --------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(256) canonical_fold_kernel(const double *__restrict__ in, int64_t n_rows, double *__restrict__ out) {
    constexpr int BINS = 1 << (2 * K);
    constexpr int PER = (BINS + 255) / 256;                            // consecutive bins per thread
    __shared__ uint16_t rep[BINS];
    __shared__ int warp_tot[8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int mine = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const uint32_t y = threadIdx.x * PER + j;
        mine += (y < (uint32_t)BINS && y <= revcomp_fast<K>(y)) ? 1 : 0;
    }
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    int base = incl - mine, n_canon = 0;
    for (int w = 0; w < 8; ++w) {
        base += w < wid ? warp_tot[w] : 0;
        n_canon += warp_tot[w];
    }
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const uint32_t y = threadIdx.x * PER + j;
        if (y < (uint32_t)BINS && y <= revcomp_fast<K>(y)) rep[base++] = (uint16_t)y;
    }
    __syncthreads();
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        const double *row = in + r * BINS;
        for (int c = lane; c < n_canon; c += 32) {
            const uint32_t y = rep[c], z = revcomp_fast<K>(y);
            out[r * n_canon + c] = (z == y) ? row[y] : row[y] + row[z];
        }
    }
}

// --------------------------------------------------------------------------------------------------
// simple cross-check kernel: one warp per contig, every lane re-reads the k bytes of its window, global atomics
// --------------------------------------------------------------------------------------------------
__device__ __forceinline__ int ref_symbol(uint8_t c) {
    return c == 'A' ? 0 : c == 'T' ? 1 : c == 'G' ? 2 : c == 'C' ? 3 : -1;
}

__global__ void kmer_naive_kernel(const uint8_t *__restrict__ seq, const int64_t *__restrict__ off, int64_t n_contigs,
                                  int k, uint32_t *__restrict__ counts, const uint16_t *__restrict__ rc_lut,
                                  const uint16_t *__restrict__ compact_lut, int out_bins) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp; c < n_contigs; c += n_warps) {
        const int64_t start = off[c], end = off[c + 1];
        for (int64_t p = start + lane; p + k <= end; p += 32) {
            uint32_t idx = 0;
            bool ok = true;
            for (int j = 0; j < k; ++j) {
                const int s = ref_symbol(seq[p + j]);
                ok &= s >= 0;
                idx = idx * 4u + (uint32_t)(s & 3);
            }
            if (!ok) continue;
            if (rc_lut) {
                const uint32_t r = rc_lut[idx];
                idx = compact_lut[r < idx ? r : idx];
            }
            atomicAdd(&counts[c * (int64_t)out_bins + idx], 1u);
        }
    }
}

// kmer.normalize_counts (scripts/kmer.py:209-221): one warp per row
__global__ void normalize_kernel(const uint32_t *__restrict__ counts, int64_t n_rows, int64_t bins, double *__restrict__ freq) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        unsigned long long total = 0;
        for (int64_t b = lane; b < bins; b += 32) total += counts[r * bins + b];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(FULL, total, d);
        const double dt = (double)total;
        for (int64_t b = lane; b < bins; b += 32) freq[r * bins + b] = (double)counts[r * bins + b] / dt;
    }
}

// --------------------------------------------------------------------------------------------------
// K1 pack: 32 bases per thread -> two code words + one validity word
// --------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t squeeze_pairs(uint32_t x) {      // one bit per 2-bit pair, order kept
    x &= 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    x = (x | (x >> 8)) & 0x0000FFFFu;
    return x;
}

__global__ void pack_kernel(const uint8_t *__restrict__ seq, int64_t n_bases, uint32_t *__restrict__ codes,
                            uint32_t *__restrict__ valid) {
    const int64_t n_groups = (n_bases + 31) >> 5;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
        uint32_t vbits = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t chunk = 2 * g + h;
            const int64_t b0 = chunk << 4;
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            int hi = 0;
            if (b0 + 16 <= n_bases) {
                const uint4 raw = ldg_stream(reinterpret_cast<const uint4 *>(seq) + chunk);
                w[0] = raw.x; w[1] = raw.y; w[2] = raw.z; w[3] = raw.w;
                hi = 16;
            } else if (b0 < n_bases) {
                hi = (int)(n_bases - b0);
                for (int i = 0; i < hi; ++i) w[i >> 2] |= (uint32_t)seq[b0 + i] << (8 * (i & 3));
            }
            if (b0 < n_bases) {
                uint32_t blank = blank_mask16_be(w) | outside_mask16_be(0, hi);
                codes[chunk] = codes16_be(w) & ~blank;
                vbits |= (~squeeze_pairs(blank) & 0xFFFFu) << (16 * (1 - h));
            }
        }
        valid[g] = vbits;
    }
}

// --------------------------------------------------------------------------------------------------
// histogram from the packed form: same warp-per-contig walk, 16 bases per lane per step
// --------------------------------------------------------------------------------------------------
template <int K, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
kmer_hist_packed_kernel(const uint32_t *__restrict__ codes, const uint32_t *__restrict__ valid,
                        const int64_t *__restrict__ off, int64_t n_contigs, uint32_t *__restrict__ counts,
                        double *__restrict__ freq, const uint16_t *__restrict__ rc_lut,
                        const uint16_t *__restrict__ compact_lut, int out_bins,
                        unsigned long long *work_counter, int contigs_per_item) {
    using Cfg = HistCfg<K, 1>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const uint32_t base = (smem_u32(smem_raw) + (uint32_t)Cfg::ALIGN - 1u) & ~((uint32_t)Cfg::ALIGN - 1u);
    const uint32_t tab = base + (uint32_t)warp * Cfg::ALIGN;
    const bool canonical = rc_lut != nullptr;
    for (int i = lane; i < Cfg::TAB_BINS; i += 32) sts_u32(tab + 4u * i, 0u);
    __syncwarp();

    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(work_counter, 1ull);
        item = __shfl_sync(FULL, item, 0);
        const int64_t first = (int64_t)item * contigs_per_item;
        if (first >= n_contigs) break;
        const int64_t last = (first + contigs_per_item < n_contigs) ? first + contigs_per_item : n_contigs;
        for (int64_t c = first; c < last; ++c) {
            const int64_t start = off[c], end = off[c + 1];
            if (end - start >= K) {
                const int64_t c0 = start >> 4;
                const int nchunks = (int)(((end + 15) >> 4) - c0);
                const int startrel = (int)(start - (c0 << 4));
                const int endrel = (int)(end - (c0 << 4));
                auto fetch = [&](int it) -> Dec {
                    const int ci = it * 32 + lane;
                    if (ci >= nchunks) return Dec{0u, 0xFFFFFFFFu};
                    const int64_t chunk = c0 + ci;
                    Dec d;
                    d.s = codes[chunk];
                    const uint32_t v16 = (valid[chunk >> 1] >> (16 * (1 - (int)(chunk & 1)))) & 0xFFFFu;
                    d.blank = 0u;
                    if (v16 != 0xFFFFu) {                       // spread 16 validity bits to blank pairs
                        uint32_t x = (~v16) & 0xFFFFu;
                        x = (x | (x << 8)) & 0x00FF00FFu;
                        x = (x | (x << 4)) & 0x0F0F0F0Fu;
                        x = (x | (x << 2)) & 0x33333333u;
                        x = (x | (x << 1)) & 0x55555555u;
                        d.blank = x | (x << 1);
                    }
                    const int pos = ci << 4;
                    if (startrel - pos > 0 || endrel - pos < 16) d.blank |= outside_mask16_be(startrel - pos, endrel - pos);
                    return d;
                };
                const int n_iter = (nchunks + 31) >> 5;
                Dec cur = fetch(0);
                for (int it = 0; it < n_iter; ++it) {
                    const Dec nxt = fetch(it + 1);
                    // the 16 bases that follow this lane's: the next lane's chunk, and for lane 31 lane 0's chunk of the NEXT step --
                    // one rotating shuffle in which lane 0 offers its next chunk (nobody needs its current one)
                    const uint32_t hi_s = __shfl_sync(FULL, lane == 0 ? nxt.s : cur.s, (lane + 1) & 31);
                    const bool dirty = (cur.blank != 0u) | ((lane == 0) & (nxt.blank != 0u));
                    if (!__any_sync(FULL, dirty)) {
#pragma unroll
                        for (int p = 0; p < 16; ++p) red_shared_inc(tab | window_offset<K>(cur.s, hi_s, p));
                    } else {
                        const uint32_t hi_b = __shfl_sync(FULL, lane == 0 ? nxt.blank : cur.blank, (lane + 1) & 31);
#pragma unroll
                        for (int p = 0; p < 16; ++p)
                            if (window_bits<K>(cur.blank, hi_b, p) == 0u) red_shared_inc(tab + window_offset<K>(cur.s, hi_s, p));
                    }
                    cur = nxt;
                }
            }
            __syncwarp();
            unsigned long long total = 0;
            for (int y = lane; y < Cfg::OUT_BINS; y += 32) total += lds_u32(tab + 4u * y);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(FULL, total, d);
            const double dtotal = (double)total;
            if (!canonical) {
                for (int y = lane; y < Cfg::OUT_BINS; y += 32) {
                    const uint32_t v = lds_u32(tab + 4u * y);
                    if (counts) counts[c * Cfg::OUT_BINS + y] = v;
                    if (freq) freq[c * Cfg::OUT_BINS + y] = (double)v / dtotal;
                }
            } else {
                for (int y = lane; y < Cfg::OUT_BINS; y += 32) {
                    const uint32_t r = rc_lut[y];
                    if (r < (uint32_t)y) {
                        const uint32_t v = lds_u32(tab + 4u * y);
                        if (v) red_shared_add(tab + 4u * r, v);
                    }
                }
                __syncwarp();
                for (int y = lane; y < Cfg::OUT_BINS; y += 32) {
                    const uint32_t r = rc_lut[y];
                    if ((uint32_t)y <= r) {
                        const uint32_t v = lds_u32(tab + 4u * y);
                        const int64_t o = c * (int64_t)out_bins + compact_lut[y];
                        if (counts) counts[o] = v;
                        if (freq) freq[o] = (double)v / dtotal;
                    }
                }
            }
            __syncwarp();
            for (int i = lane; i < Cfg::TAB_BINS; i += 32) sts_u32(tab + 4u * i, 0u);
            __syncwarp();
        }
    }
}

// --------------------------------------------------------------------------------------------------
// host-side launchers
// --------------------------------------------------------------------------------------------------
struct CountWorkspace {
    PlanHeader *plan;                // work counter + planning totals, 256-byte slot (zeroed per call)
    uint16_t *rc_lut;                // 4096 entries
    uint16_t *compact_lut;           // 4096 entries: bin -> compact canonical bin
    uint16_t *canon_lut;             // 4096 entries: compact canonical bin -> representative bin
    PlanEntry *entries;              // the list of work items (see "work plan" above), `cap` of them
    unsigned long long cap;
    unsigned long long *counter() const { return &plan->counter; }
};
static constexpr size_t kCountWorkspaceFixed = 256 + 3 * 4096 * sizeof(uint16_t);      // 24832 = 97 * 256
static_assert(kCountWorkspaceFixed % 256 == 0, "workspace layout");

static CountWorkspace carve(void *ws, size_t ws_bytes) {
    CountWorkspace w;
    unsigned char *p = static_cast<unsigned char *>(ws);
    w.plan = reinterpret_cast<PlanHeader *>(p);
    w.rc_lut = reinterpret_cast<uint16_t *>(p + 256);
    w.compact_lut = w.rc_lut + 4096;
    w.canon_lut = w.rc_lut + 8192;
    w.cap = ws_bytes > kCountWorkspaceFixed ? (ws_bytes - kCountWorkspaceFixed) / sizeof(PlanEntry) : 0;
    w.entries = reinterpret_cast<PlanEntry *>(p + kCountWorkspaceFixed);
    return w;
}

static EventRing g_hist_ring;        // brackets of the kmer_hist_kernel launches (option "time_kernels")
int kmer_hist_last_ms(float *ms) { return g_hist_ring.mean_ms(ms); }

int hist_stride_for_k4 = 2;          // tuning knob (phm_set_option)
int hist_stride_for_k5 = 0;          // 0 = automatic: 6-mers at every second base in 16-bit packed counters for plain bins (7.96 vs 8.22 ms),
                                     // plain 5-mers on the bank-swizzled table for canonical bins (7.70 vs 8.90 ms); 1 | 2 force one
int hist_warps_k6 = 13;
int hist_warps_k5 = 18;               // packed k = 5 table: one CTA of 18 warps per SM (7.79 ms) or 8 warps per CTA, 2 CTAs per SM (8.00)
int hist_tma = 0;                    // 1 = sequence staged in shared memory by TMA bulk copies (k = 4, 5, 6)
int hist_plan = 1;                   // 0 = no work plan: every contig is one item drawn in file order (round-1 scheduling)
int hist_canonical_swizzle = 1;      // k = 5, 6 canonical: bank-swizzled table + shared-memory look-up table (0 = plain layout, for comparison)

// the planning passes of one call (see "work plan"): totals per class, then the list; both read only the offset table
static int launch_plan(const int64_t *off, int64_t n, int k, const CountWorkspace &w, uint32_t *counts, double *freq, int out_bins,
                       cudaStream_t st) {
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    hist_plan_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(off, n, w.plan, RecordRanges());
    PHM_LAUNCH_CHECK();
    hist_plan_fill_kernel<<<(unsigned)blocks, 256, 0, st>>>(off, n, k, w.plan, w.entries, w.cap, counts, freq, out_bins, RecordRanges());
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

// a span call (phm_kmer_count_spans): span i of the array is row i
struct SpanList {
    const int64_t *spans; int64_t n_records;
};

// The planning passes of a span call: the count pass, which also validates every span; one synchronisation to read its totals;
// then the fill pass, only when every span is valid and the exact list fits.  *n_items: the list's length.
static int launch_span_plan(const int64_t *off, int64_t n, const SpanList &sl, int k, const CountWorkspace &w, uint32_t *counts,
                            double *freq, int out_bins, cudaStream_t st, unsigned long long *n_items) {
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const SpanRanges src{sl.spans, sl.n_records};
    PHM_CUDA_CHECK(cudaMemsetAsync(&w.plan->first_bad, 0xFF, sizeof(unsigned long long), st));
    hist_plan_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(off, n, w.plan, src);
    PHM_LAUNCH_CHECK();
    PlanHeader h;
    PHM_CUDA_CHECK(cudaMemcpyAsync(&h, w.plan, sizeof(PlanHeader), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h.first_bad != ~0ull) {
        // error path only: the span's fields, and its record's offsets when it names one
        int64_t f[3] = {0, 0, 0}, rec[2] = {0, 0};
        PHM_CUDA_CHECK(cudaMemcpyAsync(f, sl.spans + 3 * (int64_t)h.first_bad, sizeof(f), cudaMemcpyDeviceToHost, st));
        const bool named = f[0] >= 0 && f[0] < sl.n_records;
        if (named) PHM_CUDA_CHECK(cudaMemcpyAsync(rec, off + f[0], sizeof(rec), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaStreamSynchronize(st));
        const char *why = !named ? "names no record" : f[1] < 0 ? "starts before its record" : f[2] < f[1] ? "ends before it starts"
                                                                                                      : "ends past its record";
        set_error("invalid argument: span %llu (record %lld, start %lld, end %lld) %s (%lld records, this one %lld bases long)",
                  h.first_bad, (long long)f[0], (long long)f[1], (long long)f[2], why, (long long)sl.n_records,
                  (long long)(rec[1] - rec[0]));
        return PHM_E_ARG;
    }
    *n_items = h.need[0] + h.need[1] + h.need[2] + h.need[3];
    if (*n_items > w.cap) {
        set_error("workspace too small for the %lld spans: their list needs %llu items, the workspace holds %llu", (long long)n, *n_items,
                  w.cap);
        return PHM_E_WORKSPACE;
    }
    hist_plan_fill_kernel<<<(unsigned)blocks, 256, 0, st>>>(off, n, k, w.plan, w.entries, w.cap, counts, freq, out_bins, src);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

// a window call (phm_kmer_count_windows): the slice [first, first + n) of the windows of the records, rows 0 .. n - 1
struct WindowSlice {
    const int64_t *wo; int64_t n_records, window, step, first, n;
    int64_t *spans;
};

static int launch_window_plan(const int64_t *off, const WindowSlice &ws, int k, const CountWorkspace &w, uint32_t *counts,
                              double *freq, int out_bins, cudaStream_t st) {
    const uint32_t per = plan_tiles(ws.window);
    int64_t blocks = (ws.n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    window_plan_kernel<<<(unsigned)blocks, 256, 0, st>>>(off, ws.wo, ws.n_records, ws.window, ws.step, ws.first, ws.n, k, per,
                                                         per > 1u ? 0 : N_CLASS - 1, w.plan, w.entries, counts, freq, out_bins,
                                                         ws.spans);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

// win != nullptr: count the windows of a slice instead of whole records (`n` is then the slice's window count); spans != nullptr:
// count n spans.  Windows and spans always take the list, whatever option hist_plan says, because no offset table describes them
template <int K, int STRIDE, int WARPS, bool EMIT = false, bool SWZ = false, int STAGES = 0>
static int launch_hist(const uint8_t *seq, const int64_t *off, int64_t n, uint32_t *counts, double *freq,
                       const uint16_t *rc, const uint16_t *compact, int out_bins, const CountWorkspace &w,
                       cudaStream_t st, tc::QueryEmit emit = tc::QueryEmit(), const WindowSlice *win = nullptr,
                       const SpanList *spans = nullptr) {
    using Cfg = HistCfg<K, STRIDE>;
    const size_t smem = (size_t)WARPS * Cfg::WARP_BYTES + Cfg::ALIGN + (size_t)WARPS * STAGES * (STAGE_BYTES + 8);
    auto kern = kmer_hist_kernel<K, STRIDE, WARPS, EMIT, SWZ, STAGES>;
    PHM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    PHM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem));
    if (per_sm < 1) { set_error("histogram kernel does not fit on an SM (smem %zu)", smem); return PHM_E_UNSUPPORTED; }
    HistJob job;
    job.seq = seq; job.off = off; job.n_contigs = n; job.counts = counts; job.freq = freq;
    job.rc_lut = rc; job.canon_lut = compact; job.out_bins = out_bins;
    job.plan = w.plan; job.entries = w.entries;
    job.cap = (hist_plan || win || spans) ? w.cap : 0ull;
    const bool timed = g_hist_ring.begin(st);           // the bracket covers the whole counting stage: planning passes, histogram, finish
    unsigned long long span_items = 0;
    if (win) {
        const int rc_plan = launch_window_plan(off, *win, K, w, counts, freq, out_bins, st);
        if (rc_plan != PHM_OK) return rc_plan;
    } else if (spans) {
        const int rc_plan = launch_span_plan(off, n, *spans, K, w, counts, freq, out_bins, st, &span_items);
        if (rc_plan != PHM_OK) return rc_plan;
    } else if (job.cap > 0) {
        const int rc_plan = launch_plan(off, n, K, w, counts, freq, out_bins, st);
        if (rc_plan != PHM_OK) return rc_plan;
    }
    constexpr int per_item = (K >= 6) ? 4 : 1;
    int64_t grid = (int64_t)per_sm * sm_count();
    const int64_t items = win ? (n * (int64_t)plan_tiles(win->window) + per_item - 1) / per_item          // the window list, exactly
                              : spans ? ((int64_t)span_items + per_item - 1) / per_item                  // the span list, exactly
                                      : (n + (int64_t)job.cap + per_item - 1) / per_item;  // upper bound: the list can hold at most cap items
    const int64_t need = (items + WARPS - 1) / WARPS;
    if (grid > need) grid = need < 1 ? 1 : need;
    kern<<<(unsigned)grid, WARPS * 32, smem, st>>>(job, emit);
    PHM_LAUNCH_CHECK();
    if (job.cap > 0) {
        hist_finish_kernel<EMIT><<<sm_count(), 256, 0, st>>>(job, emit);
        PHM_LAUNCH_CHECK();
    }
    if (timed) g_hist_ring.end(st);
    return PHM_OK;
}

// k = 4 histogram that also emits the scorer's query operands (called by phm_count_score)
int launch_count_emit(const uint8_t *seq, const int64_t *off, int64_t n, uint32_t *counts, void *ws, size_t ws_bytes,
                      tc::QueryEmit emit, cudaStream_t st);

template <int K, int WARPS>
static int launch_hist_packed(const uint32_t *codes, const uint32_t *valid, const int64_t *off, int64_t n,
                              uint32_t *counts, double *freq, const uint16_t *rc, const uint16_t *compact,
                              int out_bins, unsigned long long *counter, cudaStream_t st) {
    using Cfg = HistCfg<K, 1>;
    const size_t smem = (size_t)WARPS * Cfg::WARP_BYTES + Cfg::ALIGN;
    auto kern = kmer_hist_packed_kernel<K, WARPS>;
    PHM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    PHM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem));
    if (per_sm < 1) { set_error("packed histogram kernel does not fit on an SM (smem %zu)", smem); return PHM_E_UNSUPPORTED; }
    int64_t grid = (int64_t)per_sm * sm_count();
    const int per_item = 4;
    const int64_t items = (n + per_item - 1) / per_item;
    const int64_t need = (items + WARPS - 1) / WARPS;
    if (grid > need) grid = need < 1 ? 1 : need;
    kern<<<(unsigned)grid, WARPS * 32, smem, st>>>(codes, valid, off, n, counts, freq, rc, compact, out_bins, counter, per_item);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

static int64_t canonical_bins(int k) {
    int64_t n = 0;
    for (uint32_t y = 0; y < (1u << (2 * k)); ++y) n += (y <= revcomp_bin(y, k));
    return n;
}

int launch_count_emit(const uint8_t *seq, const int64_t *off, int64_t n, uint32_t *counts, void *ws, size_t ws_bytes,
                      tc::QueryEmit emit, cudaStream_t st) {
    PHM_REQUIRE(seq != nullptr && off != nullptr && counts != nullptr && ws != nullptr, "null pointer");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(seq) & 15u) == 0, "d_seq must be 16-byte aligned");
    if (ws_bytes < kCountWorkspaceFixed) { set_error("count workspace too small"); return PHM_E_WORKSPACE; }
    CountWorkspace w = carve(ws, ws_bytes);
    PHM_CUDA_CHECK(cudaMemsetAsync(w.plan, 0, 256, st));
    if (hist_tma)
        return launch_hist<4, 2, 8, true, false, 4>(seq, off, n, counts, nullptr, nullptr, nullptr, 256, w, st, emit);
    return launch_hist<4, 2, 8, true>(seq, off, n, counts, nullptr, nullptr, nullptr, 256, w, st, emit);
}

}  // namespace phm

using namespace phm;

extern "C" int64_t phm_num_bins(int k, uint32_t flags) {
    if (k < 1 || k > 6) return -1;
    return (flags & PHM_COUNT_CANONICAL) ? canonical_bins(k) : ((int64_t)1 << (2 * k));
}

// Fixed part (work counter, canonical look-up tables) + the list of work items: one per contig, plus the extra tiles of contigs of
// SPLIT_MIN bases and more (at most n_bases / TILE of them).  A smaller workspace (n_bases understated) is legal: the plan is then
// switched off on the device and contigs are drawn whole, in file order.
extern "C" size_t phm_kmer_count_workspace_bytes(int64_t n_contigs, int64_t n_bases, int, uint32_t) {
    const size_t slots = (size_t)(n_contigs > 0 ? n_contigs : 0) + (size_t)(n_bases > 0 ? n_bases / TILE : 0) + 64;
    return kCountWorkspaceFixed + ((slots * sizeof(PlanEntry) + 255) & ~(size_t)255);
}

static int prepare_count(int64_t n_contigs, int k, uint32_t flags, void *ws, size_t ws_bytes, const void *offsets,
                         CountWorkspace *w, const uint16_t **rc, const uint16_t **compact, int *out_bins,
                         cudaStream_t st) {
    PHM_REQUIRE(k >= 1 && k <= 6, "k must be 1..6");
    PHM_REQUIRE(n_contigs >= 0, "n_contigs must be >= 0");
    PHM_REQUIRE(offsets != nullptr || n_contigs == 0, "d_offsets is null");
    PHM_REQUIRE(ws != nullptr, "d_workspace is null");
    if (ws_bytes < kCountWorkspaceFixed) { set_error("workspace too small: %zu < %zu", ws_bytes, kCountWorkspaceFixed); return PHM_E_WORKSPACE; }
    *w = carve(ws, ws_bytes);
    PHM_CUDA_CHECK(cudaMemsetAsync(w->plan, 0, 256, st));
    *rc = nullptr; *compact = nullptr;
    *out_bins = 1 << (2 * k);
    if (flags & PHM_COUNT_CANONICAL) {
        canonical_lut_kernel<<<1, 1024, 0, st>>>(k, w->rc_lut, w->compact_lut, w->canon_lut);
        PHM_LAUNCH_CHECK();
        *rc = w->rc_lut; *compact = w->compact_lut;
        *out_bins = (int)canonical_bins(k);
    }
    return PHM_OK;
}

// the histogram variant of k (and of the tuning options), for a call over records, over the windows of a slice or over spans
static int dispatch_hist(int k, const uint8_t *seq, const int64_t *off, int64_t n, uint32_t *counts, double *freq, const uint16_t *rc,
                         const uint16_t *canon, int out_bins, const CountWorkspace &w, cudaStream_t st, const WindowSlice *win,
                         const SpanList *sp = nullptr) {
    const tc::QueryEmit e = tc::QueryEmit();
    switch (k) {
        case 1: return launch_hist<1, 1, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
        case 2: return launch_hist<2, 1, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
        case 3: return launch_hist<3, 1, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
        case 4:
            if (hist_stride_for_k4 == 2)
                return hist_tma ? launch_hist<4, 2, 8, false, false, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp)
                                : launch_hist<4, 2, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            return launch_hist<4, 1, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
        case 5:
            if ((hist_stride_for_k5 == 2 || (hist_stride_for_k5 == 0 && !rc)) && hist_warps_k5 == 18)
                return launch_hist<5, 2, 18>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            if (hist_stride_for_k5 == 2 || (hist_stride_for_k5 == 0 && !rc))
                return launch_hist<5, 2, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            if (rc && hist_canonical_swizzle)
                return hist_tma ? launch_hist<5, 1, 8, false, true, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp)
                                : launch_hist<5, 1, 8, false, true>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            return hist_tma ? launch_hist<5, 1, 8, false, false, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp)
                            : launch_hist<5, 1, 8>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
        case 6:
            if (hist_warps_k6 == 4)
                return launch_hist<6, 1, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            if (rc && hist_canonical_swizzle)
                return hist_tma ? launch_hist<6, 1, 11, false, true, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp)
                                : launch_hist<6, 1, 13, false, true>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
            return hist_tma ? launch_hist<6, 1, 11, false, false, 4>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp)
                            : launch_hist<6, 1, 13>(seq, off, n, counts, freq, rc, canon, out_bins, w, st, e, win, sp);
    }
    return PHM_E_ARG;
}

extern "C" int phm_kmer_count(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_contigs, int k, uint32_t flags,
                              uint32_t *d_counts, double *d_freq, void *d_workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CountWorkspace w; const uint16_t *rc, *compact; int out_bins;
    int rcode = prepare_count(n_contigs, k, flags, d_workspace, workspace_bytes, d_offsets, &w, &rc, &compact, &out_bins, st);
    if (rcode != PHM_OK) return rcode;
    if (n_contigs == 0) return PHM_OK;
    PHM_REQUIRE(d_seq != nullptr, "d_seq is null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_seq) & 15u) == 0, "d_seq must be 16-byte aligned");
    PHM_REQUIRE(d_counts != nullptr || d_freq != nullptr, "both outputs are null");

    const uint16_t *canon = rc ? w.canon_lut : nullptr;           // compact bin -> representative (the histogram kernel gathers)
    if (flags & PHM_COUNT_NAIVE) {
        PHM_REQUIRE(d_counts != nullptr, "the naive kernel needs d_counts");
        PHM_CUDA_CHECK(cudaMemsetAsync(d_counts, 0, (size_t)n_contigs * out_bins * sizeof(uint32_t), st));
        int64_t blocks = (n_contigs + 7) / 8;
        if (blocks > 148 * 16) blocks = 148 * 16;
        kmer_naive_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_seq, d_offsets, n_contigs, k, d_counts, rc, compact, out_bins);
        PHM_LAUNCH_CHECK();
        if (d_freq) return phm_normalize_counts(d_counts, n_contigs, out_bins, d_freq, stream);
        return PHM_OK;
    }
    return dispatch_hist(k, d_seq, d_offsets, n_contigs, d_counts, d_freq, rc, canon, out_bins, w, st, nullptr);
}

extern "C" int phm_window_offsets(const int64_t *d_offsets, int64_t n_records, int64_t window, int64_t step, int64_t *d_window_offsets,
                                  void *stream) {
    PHM_REQUIRE(window >= 1 && step >= 1, "window and step must be >= 1");
    PHM_REQUIRE(n_records >= 0, "n_records must be >= 0");
    PHM_REQUIRE(d_window_offsets != nullptr && (d_offsets != nullptr || n_records == 0), "null pointer");
    PHM_REQUIRE(((reinterpret_cast<uintptr_t>(d_offsets) | reinterpret_cast<uintptr_t>(d_window_offsets)) & 7u) == 0,
                "offsets must be 8-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_records == 0) {
        PHM_CUDA_CHECK(cudaMemsetAsync(d_window_offsets, 0, sizeof(int64_t), st));
        return PHM_OK;
    }
    const int64_t tiles = (n_records + WO_TILE - 1) / WO_TILE;
    window_offsets_kernel<<<(unsigned)tiles, 256, 0, st>>>(d_offsets, n_records, window, step, d_window_offsets);
    PHM_LAUNCH_CHECK();
    if (tiles > 1) {
        window_offsets_carry_kernel<<<1, 1024, 0, st>>>(n_records, d_window_offsets);
        PHM_LAUNCH_CHECK();
        int64_t blocks = (n_records - WO_TILE + 255) / 256;
        if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
        window_offsets_add_kernel<<<(unsigned)blocks, 256, 0, st>>>(n_records, d_window_offsets);
        PHM_LAUNCH_CHECK();
    }
    return PHM_OK;
}

extern "C" size_t phm_kmer_count_windows_workspace_bytes(int64_t n_windows, int64_t window, int, uint32_t) {
    const size_t slots = (size_t)(n_windows > 0 ? n_windows : 0) * plan_tiles(window > 0 ? window : 1);
    return kCountWorkspaceFixed + ((slots * sizeof(PlanEntry) + 255) & ~(size_t)255);
}

extern "C" int phm_kmer_count_windows(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_records, const int64_t *d_window_offsets,
                                      int64_t window, int64_t step, int64_t first_window, int64_t n_windows, int k, uint32_t flags,
                                      uint32_t *d_counts, double *d_freq, int64_t *d_spans, void *d_workspace, size_t workspace_bytes,
                                      void *stream) {
    // every argument is checked before the device is touched
    PHM_REQUIRE(k >= 1 && k <= 6, "k must be 1..6");
    PHM_REQUIRE(window >= 1 && step >= 1, "window and step must be >= 1");
    PHM_REQUIRE((flags & ~PHM_COUNT_CANONICAL) == 0u, "flags: PHM_COUNT_CANONICAL is the only flag of a window call");
    PHM_REQUIRE(n_records >= 0, "n_records must be >= 0");
    PHM_REQUIRE(first_window >= 0 && n_windows >= 0, "first_window and n_windows must be >= 0");
    PHM_REQUIRE(n_records > 0 || first_window + n_windows == 0, "the slice lies outside the windows");
    if (n_windows == 0) return PHM_OK;
    PHM_REQUIRE(d_seq != nullptr && d_offsets != nullptr && d_window_offsets != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_counts != nullptr || d_freq != nullptr, "both outputs are null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_seq) & 15u) == 0, "d_seq must be 16-byte aligned");
    PHM_REQUIRE(((reinterpret_cast<uintptr_t>(d_offsets) | reinterpret_cast<uintptr_t>(d_window_offsets) |
                  reinterpret_cast<uintptr_t>(d_freq) | reinterpret_cast<uintptr_t>(d_spans)) & 7u) == 0 &&
                (reinterpret_cast<uintptr_t>(d_counts) & 3u) == 0, "misaligned pointer");
    const unsigned long long slots = (unsigned long long)n_windows * plan_tiles(window);
    if (workspace_bytes < kCountWorkspaceFixed || (workspace_bytes - kCountWorkspaceFixed) / sizeof(PlanEntry) < slots) {
        set_error("workspace too small for %lld windows: %zu < %zu bytes", (long long)n_windows, workspace_bytes,
                  phm_kmer_count_windows_workspace_bytes(n_windows, window, k, flags));
        return PHM_E_WORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int64_t total = 0;                                                  // the slice must lie inside [0, total windows)
    PHM_CUDA_CHECK(cudaMemcpyAsync(&total, d_window_offsets + n_records, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (first_window > total || n_windows > total - first_window) {
        set_error("invalid argument: windows [%lld, %lld) lie outside the %lld windows of the records", (long long)first_window,
                  (long long)(first_window + n_windows), (long long)total);
        return PHM_E_ARG;
    }
    CountWorkspace w; const uint16_t *rc, *compact; int out_bins;
    int rcode = prepare_count(n_windows, k, flags, d_workspace, workspace_bytes, d_offsets, &w, &rc, &compact, &out_bins, st);
    if (rcode != PHM_OK) return rcode;
    const WindowSlice win{d_window_offsets, n_records, window, step, first_window, n_windows, d_spans};
    return dispatch_hist(k, d_seq, d_offsets, n_windows, d_counts, d_freq, rc, rc ? w.canon_lut : nullptr, out_bins, w, st, &win);
}

// Fixed part + one list item per span, plus the extra tiles of spans of SPLIT_MIN bases and more (at most n_span_bases / TILE).
extern "C" size_t phm_kmer_count_spans_workspace_bytes(int64_t n_spans, int64_t n_span_bases, int, uint32_t) {
    const size_t slots = (size_t)(n_spans > 0 ? n_spans : 0) + (size_t)(n_span_bases > 0 ? n_span_bases / TILE : 0);
    return kCountWorkspaceFixed + ((slots * sizeof(PlanEntry) + 255) & ~(size_t)255);
}

extern "C" int phm_kmer_count_spans(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_records, const int64_t *d_spans,
                                    int64_t n_spans, int k, uint32_t flags, uint32_t *d_counts, double *d_freq, void *d_workspace,
                                    size_t workspace_bytes, void *stream) {
    // every argument is checked before the device is touched; the spans themselves are checked by the count pass
    PHM_REQUIRE(k >= 1 && k <= 6, "k must be 1..6");
    PHM_REQUIRE((flags & ~PHM_COUNT_CANONICAL) == 0u, "flags: PHM_COUNT_CANONICAL is the only flag of a span call");
    PHM_REQUIRE(n_records >= 0 && n_spans >= 0, "n_records and n_spans must be >= 0");
    if (n_spans == 0) return PHM_OK;
    PHM_REQUIRE(d_seq != nullptr && d_offsets != nullptr && d_spans != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_counts != nullptr || d_freq != nullptr, "both outputs are null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_seq) & 15u) == 0, "d_seq must be 16-byte aligned");
    PHM_REQUIRE(((reinterpret_cast<uintptr_t>(d_offsets) | reinterpret_cast<uintptr_t>(d_spans) | reinterpret_cast<uintptr_t>(d_freq)) & 7u) == 0 &&
                (reinterpret_cast<uintptr_t>(d_counts) & 3u) == 0, "misaligned pointer");
    if (workspace_bytes < kCountWorkspaceFixed || (workspace_bytes - kCountWorkspaceFixed) / sizeof(PlanEntry) < (unsigned long long)n_spans) {
        set_error("workspace too small for %lld spans: %zu < %zu bytes", (long long)n_spans, workspace_bytes,
                  phm_kmer_count_spans_workspace_bytes(n_spans, 0, k, flags));
        return PHM_E_WORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CountWorkspace w; const uint16_t *rc, *compact; int out_bins;
    int rcode = prepare_count(n_spans, k, flags, d_workspace, workspace_bytes, d_offsets, &w, &rc, &compact, &out_bins, st);
    if (rcode != PHM_OK) return rcode;
    const SpanList sl{d_spans, n_records};
    return dispatch_hist(k, d_seq, d_offsets, n_spans, d_counts, d_freq, rc, rc ? w.canon_lut : nullptr, out_bins, w, st, nullptr, &sl);
}

extern "C" int phm_kmer_count_packed(const uint32_t *d_codes, const uint32_t *d_valid, const int64_t *d_offsets,
                                     int64_t n_contigs, int k, uint32_t flags, uint32_t *d_counts, double *d_freq,
                                     void *d_workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CountWorkspace w; const uint16_t *rc, *compact; int out_bins;
    int rcode = prepare_count(n_contigs, k, flags, d_workspace, workspace_bytes, d_offsets, &w, &rc, &compact, &out_bins, st);
    if (rcode != PHM_OK) return rcode;
    if (n_contigs == 0) return PHM_OK;
    PHM_REQUIRE(d_codes != nullptr && d_valid != nullptr, "packed inputs are null");
    PHM_REQUIRE(d_counts != nullptr || d_freq != nullptr, "both outputs are null");
    switch (k) {
        case 1: return launch_hist_packed<1, 8>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
        case 2: return launch_hist_packed<2, 8>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
        case 3: return launch_hist_packed<3, 8>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
        case 4: return launch_hist_packed<4, 8>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
        case 5: return launch_hist_packed<5, 8>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
        case 6: return launch_hist_packed<6, 4>(d_codes, d_valid, d_offsets, n_contigs, d_counts, d_freq, rc, compact, out_bins, w.counter(), st);
    }
    return PHM_E_ARG;
}

extern "C" int phm_normalize_counts(const uint32_t *d_counts, int64_t n_rows, int64_t bins, double *d_freq, void *stream) {
    PHM_REQUIRE(n_rows >= 0 && bins > 0, "bad shape");
    if (n_rows == 0) return PHM_OK;
    PHM_REQUIRE(d_counts != nullptr && d_freq != nullptr, "null pointer");
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    normalize_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_counts, n_rows, bins, d_freq);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_canonical_fold(const double *d_rows, int64_t n_rows, int k, double *d_out, void *stream) {
    PHM_REQUIRE(k >= 1 && k <= 6, "k must be 1..6");
    PHM_REQUIRE(n_rows >= 0, "n_rows must be >= 0");
    if (n_rows == 0) return PHM_OK;
    PHM_REQUIRE(d_rows != nullptr && d_out != nullptr, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
    switch (k) {
        case 1: canonical_fold_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
        case 2: canonical_fold_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
        case 3: canonical_fold_kernel<3><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
        case 4: canonical_fold_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
        case 5: canonical_fold_kernel<5><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
        default: canonical_fold_kernel<6><<<(unsigned)blocks, 256, 0, st>>>(d_rows, n_rows, d_out); break;
    }
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_pack_fasta(const uint8_t *d_seq, int64_t n_bases, uint32_t *d_codes, uint32_t *d_valid, void *stream) {
    PHM_REQUIRE(n_bases >= 0, "n_bases must be >= 0");
    if (n_bases == 0) return PHM_OK;
    PHM_REQUIRE(d_seq != nullptr && d_codes != nullptr && d_valid != nullptr, "null pointer");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_seq) & 15u) == 0, "d_seq must be 16-byte aligned");
    const int64_t groups = (n_bases + 31) >> 5;
    int64_t blocks = (groups + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 32;
    if (blocks > cap) blocks = cap;
    pack_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_seq, n_bases, d_codes, d_valid);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}
