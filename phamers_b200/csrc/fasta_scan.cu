// FASTA ingest on the device (SURVEY.md 8(f) rank 3): raw file bytes -> sequence bytes laid end to end + record offsets + header
// positions, i.e. the tokenisation kmer.count_file gets from Bio.SeqIO (reference scripts/kmer.py:131-139, scripts/fileIO.py:28-42)
// and that phamers_b200/fileIO.py::split_fasta_bytes restates on the host.
//
// Semantics (Bio.SeqIO FASTA parser over a text-mode handle, as the reference uses it): a line ends at '\n', '\r' or "\r\n"
// (universal newlines); a record starts at a line whose first byte is '>'; its sequence is every following line up to the next such
// line, with line feeds, carriage returns and blanks removed -- k-mers span line breaks but never records; text before the first '>'
// is ignored.  Tab / VT / FF / 0x1C-0x1F are stripped by the reference only at line ends (str.rstrip), which this scan does not
// model: it reports any control byte other than '\n' '\r' (result[2]) and the caller takes the exact host path for such (rare) files.
// The input allocation is readable up to the next multiple of 16 bytes; what those padding bytes hold does not matter, they read as
// '\n'.
//
// Every byte is in one of three line states: 0 = preamble (no header seen yet), 1 = inside a header line, 2 = inside a sequence line.
// A line start (first byte of the file, or the byte after '\n' or '\r') moves the state: '>' -> 1; anything else: 1 -> 2, 0 and 2
// stay.  So the '\n' of "\r\n" starts an empty line, which keeps nothing and moves 1 -> 2 as the next real line would: LF and CRLF
// files give the same outputs as with '\n' alone as the line end.
// A byte is KEPT iff its state is 2 and it is none of '\n' '\r' ' '.  The state of a byte depends on everything before it, so the
// scan works on state MAPS (3 states -> 3 states, 6 bits), whose composition is associative:
//   pass 1  fasta_tile_kernel    per 16 KB tile: its map, the kept count for each incoming state, its number of header starts
//   pass 2  fasta_chain_kernel   one CTA: exclusive scan over the tiles -> incoming state, sequence offset and record index of each tile
//   pass 3  fasta_emit_kernel    per tile, state now known: compacts the kept bytes in shared memory and writes them as whole
//                                16-byte words; writes offsets[r], header_pos[r] for the records that start in the tile
// A thread's 16 bytes are classified four at a time into 16-bit masks (SWAR zero-byte tests); the state machine then only visits
// the line starts, of which a thread usually has none or one.
// Traffic: the file is read twice and the sequence written once (~3 bytes per input byte); pass 2 touches 32 bytes per tile.
#include "phm_common.cuh"

namespace phm {
namespace fasta {

constexpr int TILE_THREADS = 1024;
constexpr int PER_THREAD = 16;
constexpr int TILE_BYTES = TILE_THREADS * PER_THREAD;      // 16 KB
constexpr int NWARPS = TILE_THREADS / 32;
static_assert(NWARPS <= 32, "one warp scans the per-warp partial results");

struct TileSummary {               // 32 bytes
    uint32_t map;                  // incoming state s -> outgoing state, 2 bits each
    uint32_t n_headers;            // header starts in the tile
    uint32_t kept[3];              // kept bytes of the tile for incoming state 0 / 1 / 2
    uint32_t odd;                  // tab / VT / FF seen
    uint32_t pad[2];
};
struct TileStart {                 // 24 bytes, written by pass 2
    int64_t seq_base;              // kept bytes before the tile
    int64_t rec_base;              // header starts before the tile
    uint32_t state;                // incoming state
    uint32_t pad;
};

constexpr uint32_t MAP_ID = 0u | (1u << 2) | (2u << 4);
__device__ __forceinline__ uint32_t map_apply(uint32_t m, uint32_t s) { return (m >> (2 * s)) & 3u; }
__device__ __forceinline__ uint32_t map_then(uint32_t first, uint32_t second) {       // s -> second(first(s))
    return map_apply(second, map_apply(first, 0)) | (map_apply(second, map_apply(first, 1)) << 2) |
           (map_apply(second, map_apply(first, 2)) << 4);
}
// ---- 16 bytes -> 16-bit class masks, four bytes at a time (SWAR) ----
// 0x80 in every byte of x that is zero
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
    return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
}
// bits 7, 15, 23, 31 -> bits 0..3 (the partial products land on distinct bits, so there are no carries)
__device__ __forceinline__ uint32_t gather4(uint32_t z) { return (((z >> 7) * 0x00204081u) >> 21) & 0xFu; }

struct Masks {
    uint32_t nl;      // byte ends a line: '\n' or '\r' (bytes at or past the end of the file count as '\n')
    uint32_t keep;    // byte is none of '\n' '\r' ' '
    uint32_t odd;     // non-zero: a control byte other than '\n' '\r' (tab / VT / FF / 0x1C-0x1F among them) is present
    uint32_t w[4];    // the bytes themselves, those past the end of the file replaced by '\n'
};

__device__ __forceinline__ Masks classify16(const uint8_t *raw, int64_t n, int64_t i0) {
    Masks m;
    m.nl = 0xFFFFu; m.keep = 0u; m.odd = 0u;
    m.w[0] = m.w[1] = m.w[2] = m.w[3] = 0x0A0A0A0Au;
    if (i0 >= n) return m;
    const uint4 v = *reinterpret_cast<const uint4 *>(raw + i0);
    m.w[0] = v.x; m.w[1] = v.y; m.w[2] = v.z; m.w[3] = v.w;
    uint32_t nl = 0u, drop = 0u;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t z_nl = zero_bytes(m.w[q] ^ 0x0A0A0A0Au), z_cr = zero_bytes(m.w[q] ^ 0x0D0D0D0Du), z_sp = zero_bytes(m.w[q] ^ 0x20202020u);
        const uint32_t z_ctrl = zero_bytes(m.w[q] & 0xE0E0E0E0u);                    // bytes 0..31
        nl |= gather4(z_nl | z_cr) << (4 * q);
        drop |= gather4(z_nl | z_cr | z_sp) << (4 * q);
        m.odd |= z_ctrl & ~(z_nl | z_cr);
    }
    m.nl = nl;
    m.keep = ~drop & 0xFFFFu;
    if (i0 + PER_THREAD > n) {                   // last chunk of the file: the bytes past the end are caller padding of any content;
        const int n_valid = (int)(n - i0);       // they are replaced by '\n', so no later reader (header_starts, byte_at, s_bytes) sees them
        const uint32_t valid = (1u << n_valid) - 1u;
        m.nl = (m.nl & valid) | (~valid & 0xFFFFu);
        m.keep &= valid;
        m.odd = 0u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int v = n_valid - 4 * q;                           // valid bytes of word q
            const uint32_t lo = v <= 0 ? 0u : (v >= 4 ? 0xFFFFFFFFu : (1u << (8 * v)) - 1u);
            m.w[q] = (m.w[q] & lo) | (0x0A0A0A0Au & ~lo);
        }
        for (int j = 0; j < n_valid; ++j) {
            const uint32_t c = (m.w[j >> 2] >> (8 * (j & 3))) & 255u;
            m.odd |= (c < 32u && c != 10u && c != 13u) ? 1u : 0u;
        }
    }
    return m;
}
// byte j (0..15) of the chunk
__device__ __forceinline__ uint32_t byte_at(const Masks &m, int j) {
    const uint32_t lo = (j & 4) ? m.w[1] : m.w[0], hi = (j & 4) ? m.w[3] : m.w[2];
    return (((j & 8) ? hi : lo) >> (8 * (j & 3))) & 255u;
}
// line starts of this thread's 16 bytes: the byte after a '\n' or '\r' (the first byte of the file starts a line)
__device__ __forceinline__ uint32_t line_starts(const uint8_t *raw, int64_t n, int64_t i0, uint32_t nl) {
    const uint32_t prev = (i0 == 0 || i0 > n) ? 10u : raw[i0 - 1];
    const uint32_t prev_nl = (prev == 10u || prev == 13u) ? 1u : 0u;
    return ((nl << 1) | prev_nl) & 0xFFFFu;
}
// which line starts are header starts ('>' as first byte of the line)
__device__ __forceinline__ uint32_t header_starts(const Masks &m, uint32_t ls) {
    uint32_t hs = 0u;
    for (uint32_t rest = ls; rest; rest &= rest - 1u) {
        const int b = __ffs(rest) - 1;
        hs |= (byte_at(m, b) == (uint32_t)'>') ? (1u << b) : 0u;
    }
    return hs;
}
// bits below the lowest set bit of `rest` (all 16 if there is none)
__device__ __forceinline__ uint32_t below_next(uint32_t rest) { return rest ? ((1u << (__ffs(rest) - 1)) - 1u) : 0xFFFFu; }

// ---------------- pass 1 ----------------
__global__ void __launch_bounds__(TILE_THREADS) fasta_tile_kernel(const uint8_t *__restrict__ raw, int64_t n, int64_t n_tiles,
                                                                  TileSummary *__restrict__ tiles) {
    __shared__ uint32_t s_map[32], s_pre[32], s_whole;
    __shared__ uint32_t s_sum[NWARPS][5];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t i0 = tile * TILE_BYTES + (int64_t)threadIdx.x * PER_THREAD;
        const Masks m = classify16(raw, n, i0);
        const uint32_t ls = line_starts(raw, n, i0, m.nl), hs = header_starts(m, ls);
        // thread-local: outgoing state and kept bytes for each incoming state; the state only changes at line starts
        uint32_t st[3] = {0u, 1u, 2u}, kept[3] = {0u, 0u, 0u};
        uint32_t rest = ls;
        kept[2] = __popc(m.keep & below_next(rest));
        while (rest) {
            const int b = __ffs(rest) - 1;
            rest &= rest - 1u;
            const uint32_t cnt = __popc(m.keep & below_next(rest) & ~((1u << b) - 1u));
            const bool is_h = (hs >> b) & 1u;
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                st[s] = is_h ? 1u : (st[s] == 1u ? 2u : st[s]);
                kept[s] += st[s] == 2u ? cnt : 0u;
            }
        }
        uint32_t heads = __popc(hs), odd = m.odd ? 1u : 0u;
        // exclusive scan of the maps over the tile: which state each thread starts in, for each state the tile may start in
        uint32_t incl = st[0] | (st[1] << 2) | (st[2] << 4);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl = map_then(up, incl);
        }
        uint32_t excl = __shfl_up_sync(FULL, incl, 1);
        if (lane == 0) excl = MAP_ID;
        __syncthreads();                                           // previous tile's shared memory is no longer read
        if (lane == 31) s_map[warp] = incl;
        __syncthreads();
        if (warp == 0) {                                           // scan of the warps' maps by one warp
            const uint32_t wm = lane < NWARPS ? s_map[lane] : MAP_ID;
            uint32_t wi = wm;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(FULL, wi, o);
                if (lane >= o) wi = map_then(up, wi);
            }
            uint32_t we = __shfl_up_sync(FULL, wi, 1);
            if (lane == 0) we = MAP_ID;
            s_pre[lane] = we;
            if (lane == 31) s_whole = wi;
        }
        __syncthreads();
        const uint32_t start = map_then(s_pre[warp], excl);        // tile's incoming state -> this thread's incoming state
        uint32_t k0 = kept[map_apply(start, 0)], k1 = kept[map_apply(start, 1)], k2 = kept[map_apply(start, 2)];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            k0 += __shfl_xor_sync(FULL, k0, o); k1 += __shfl_xor_sync(FULL, k1, o); k2 += __shfl_xor_sync(FULL, k2, o);
            heads += __shfl_xor_sync(FULL, heads, o); odd |= __shfl_xor_sync(FULL, odd, o);
        }
        if (lane == 0) { s_sum[warp][0] = k0; s_sum[warp][1] = k1; s_sum[warp][2] = k2; s_sum[warp][3] = heads; s_sum[warp][4] = odd; }
        __syncthreads();
        if (warp == 0) {
            uint32_t v0 = 0u, v1 = 0u, v2 = 0u, v3 = 0u, v4 = 0u;
            if (lane < NWARPS) { v0 = s_sum[lane][0]; v1 = s_sum[lane][1]; v2 = s_sum[lane][2]; v3 = s_sum[lane][3]; v4 = s_sum[lane][4]; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                v0 += __shfl_xor_sync(FULL, v0, o); v1 += __shfl_xor_sync(FULL, v1, o); v2 += __shfl_xor_sync(FULL, v2, o);
                v3 += __shfl_xor_sync(FULL, v3, o); v4 |= __shfl_xor_sync(FULL, v4, o);
            }
            if (lane == 0) {
                TileSummary t;
                t.map = s_whole; t.n_headers = v3; t.kept[0] = v0; t.kept[1] = v1; t.kept[2] = v2; t.odd = v4; t.pad[0] = t.pad[1] = 0u;
                tiles[tile] = t;
            }
        }
    }
}

// ---------------- pass 2: one CTA chains the tiles ----------------
// Warp w owns a contiguous range of tiles and walks it 32 tiles at a time (lane = tile: coalesced loads, warp-shuffle scans), three
// times: the range as one map; its totals once the state it starts in is known; every tile's start.
// result[0] = records, [1] = sequence bytes kept, [2] = 1 if a control byte other than '\n' '\r' was seen, [3] = tiles
__global__ void __launch_bounds__(1024) fasta_chain_kernel(const TileSummary *__restrict__ tiles, int64_t n_tiles,
                                                           TileStart *__restrict__ starts, int64_t *__restrict__ result) {
    __shared__ uint32_t s_map[32];
    __shared__ unsigned long long s_k[32], s_h[32];
    __shared__ uint32_t s_odd;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t per = ((n_tiles + 31) / 32 + 31) / 32 * 32;        // tiles per warp, a multiple of 32
    const int64_t lo = (int64_t)warp * per < n_tiles ? (int64_t)warp * per : n_tiles;
    const int64_t hi = (lo + per < n_tiles) ? lo + per : n_tiles;
    if (threadIdx.x == 0) s_odd = 0u;
    __syncthreads();
    uint32_t range_map = MAP_ID, odd = 0u;
    for (int64_t t0 = lo; t0 < hi; t0 += 32) {
        const int64_t t = t0 + lane;
        uint32_t mp = MAP_ID;
        if (t < hi) { mp = tiles[t].map; odd |= tiles[t].odd; }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(FULL, mp, o);
            if (lane >= o) mp = map_then(up, mp);
        }
        range_map = map_then(range_map, __shfl_sync(FULL, mp, 31));
    }
    if (__any_sync(FULL, odd != 0u) && lane == 0) atomicOr(&s_odd, 1u);
    if (lane == 0) s_map[warp] = range_map;
    __syncthreads();
    uint32_t before = MAP_ID;
    for (int w = 0; w < warp; ++w) before = map_then(before, s_map[w]);
    const uint32_t state0 = map_apply(before, 0u);                    // the file starts in the preamble state
    unsigned long long base_k = 0, base_h = 0;
    for (int pass = 0; pass < 2; ++pass) {
        uint32_t st_in = state0;
        unsigned long long run_k = base_k, run_h = base_h;
        for (int64_t t0 = lo; t0 < hi; t0 += 32) {
            const int64_t t = t0 + lane;
            TileSummary s;
            s.map = MAP_ID; s.n_headers = 0u; s.kept[0] = s.kept[1] = s.kept[2] = 0u;
            if (t < hi) s = tiles[t];
            uint32_t mp = s.map;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(FULL, mp, o);
                if (lane >= o) mp = map_then(up, mp);
            }
            uint32_t ex = __shfl_up_sync(FULL, mp, 1);
            if (lane == 0) ex = MAP_ID;
            const uint32_t my_state = map_apply(ex, st_in);
            const unsigned long long mk = my_state == 0u ? s.kept[0] : (my_state == 1u ? s.kept[1] : s.kept[2]), mh = s.n_headers;
            unsigned long long k = mk, h = mh;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long uk = __shfl_up_sync(FULL, k, o), uh = __shfl_up_sync(FULL, h, o);
                if (lane >= o) { k += uk; h += uh; }
            }
            if (pass == 1 && t < hi) {
                TileStart out;
                out.seq_base = (int64_t)(run_k + k - mk); out.rec_base = (int64_t)(run_h + h - mh); out.state = my_state; out.pad = 0u;
                starts[t] = out;
            }
            run_k += __shfl_sync(FULL, k, 31);
            run_h += __shfl_sync(FULL, h, 31);
            st_in = map_apply(__shfl_sync(FULL, mp, 31), st_in);
        }
        if (pass == 0) {
            if (lane == 0) { s_k[warp] = run_k; s_h[warp] = run_h; }
            __syncthreads();
            for (int w = 0; w < warp; ++w) { base_k += s_k[w]; base_h += s_h[w]; }
            if (threadIdx.x == 1023) {
                unsigned long long tk = 0, th = 0;
                for (int w = 0; w < 32; ++w) { tk += s_k[w]; th += s_h[w]; }
                result[0] = (int64_t)th; result[1] = (int64_t)tk; result[2] = (int64_t)s_odd; result[3] = n_tiles;
            }
        }
    }
}

// ---------------- pass 3 ----------------
__global__ void __launch_bounds__(TILE_THREADS) fasta_emit_kernel(const uint8_t *__restrict__ raw, int64_t n, int64_t n_tiles,
                                                                  const TileStart *__restrict__ starts, const int64_t *__restrict__ result,
                                                                  uint8_t *__restrict__ seq, int64_t *__restrict__ offsets,
                                                                  int64_t *__restrict__ header_pos, int64_t max_records) {
    __shared__ uint32_t s_map[32], s_pre[32], s_k[32], s_h[32], s_total;
    __shared__ __align__(16) uint8_t s_bytes[TILE_BYTES + 16];              // + one word of slack for the funnel shift's look-ahead
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0 && result[0] <= max_records) offsets[result[0]] = result[1];   // closing offset
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileStart ts = starts[tile];
        const int64_t i0 = tile * TILE_BYTES + (int64_t)threadIdx.x * PER_THREAD;
        const Masks m = classify16(raw, n, i0);
        const uint32_t ls = line_starts(raw, n, i0, m.nl), hs = header_starts(m, ls);
        // 1. this thread's map, to find the state it starts in
        uint32_t st[3] = {0u, 1u, 2u};
        for (uint32_t rest = ls; rest; rest &= rest - 1u) {
            const bool is_h = (hs >> (__ffs(rest) - 1)) & 1u;
#pragma unroll
            for (int s = 0; s < 3; ++s) st[s] = is_h ? 1u : (st[s] == 1u ? 2u : st[s]);
        }
        uint32_t incl = st[0] | (st[1] << 2) | (st[2] << 4);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl = map_then(up, incl);
        }
        uint32_t excl = __shfl_up_sync(FULL, incl, 1);
        if (lane == 0) excl = MAP_ID;
        __syncthreads();                                           // previous tile done with shared memory
        if (lane == 31) s_map[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t wi = lane < NWARPS ? s_map[lane] : MAP_ID;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(FULL, wi, o);
                if (lane >= o) wi = map_then(up, wi);
            }
            uint32_t we = __shfl_up_sync(FULL, wi, 1);
            if (lane == 0) we = MAP_ID;
            s_pre[lane] = we;
        }
        __syncthreads();
        uint32_t state = map_apply(map_then(s_pre[warp], excl), ts.state);
        // 2. kept bytes of this thread, with the real state
        uint32_t rest = ls;
        uint32_t keep_mask = state == 2u ? (m.keep & below_next(rest)) : 0u;
        while (rest) {
            const int b = __ffs(rest) - 1;
            rest &= rest - 1u;
            state = ((hs >> b) & 1u) ? 1u : (state == 1u ? 2u : state);
            if (state == 2u) keep_mask |= m.keep & below_next(rest) & ~((1u << b) - 1u);
        }
        const uint32_t nk = __popc(keep_mask), nh = __popc(hs);
        uint32_t ki = nk, hi = nh;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t uk = __shfl_up_sync(FULL, ki, o), uh = __shfl_up_sync(FULL, hi, o);
            if (lane >= o) { ki += uk; hi += uh; }
        }
        if (lane == 31) { s_k[warp] = ki; s_h[warp] = hi; }
        __syncthreads();
        if (warp == 0) {                                           // exclusive sums over the warps, and the tile total
            const uint32_t wk = lane < NWARPS ? s_k[lane] : 0u, wh = lane < NWARPS ? s_h[lane] : 0u;
            uint32_t sk = wk, sh2 = wh;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t uk = __shfl_up_sync(FULL, sk, o), uh = __shfl_up_sync(FULL, sh2, o);
                if (lane >= o) { sk += uk; sh2 += uh; }
            }
            s_k[lane] = sk - wk; s_h[lane] = sh2 - wh;
            if (lane == 31) s_total = sk;
        }
        __syncthreads();
        const uint32_t kpos = ki - nk + s_k[warp], hpos = hi - nh + s_h[warp];
        // 3. records that start here: offset = kept bytes before the header, position of its '>'.  With max_records < records,
        //    offsets[max_records] is the start of the first dropped record, which is where the last kept one ends.
        int64_t r = ts.rec_base + hpos;
        for (uint32_t hm = hs; hm; hm &= hm - 1u, ++r) {
            const int j = __ffs(hm) - 1;
            if (r <= max_records) offsets[r] = ts.seq_base + kpos + __popc(keep_mask & ((1u << j) - 1u));
            if (r < max_records) header_pos[r] = i0 + j;
        }
        // 4. the kept bytes: compacted in shared memory, then written as whole 16-byte words (a byte store costs a full 32-byte sector
        //    transaction in L2, and that -- not DRAM -- bounded the first version of this kernel)
        {
            uint32_t at = kpos;
#pragma unroll
            for (int j = 0; j < PER_THREAD; ++j)
                if ((keep_mask >> j) & 1u) s_bytes[at++] = (uint8_t)(m.w[j >> 2] >> (8 * (j & 3)));
        }
        __syncthreads();
        {
            const uint32_t tile_kept = s_total;
            uint8_t *dst = seq + ts.seq_base;
            uint32_t head = (uint32_t)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u);
            if (head > tile_kept) head = tile_kept;
            const uint32_t n16 = (tile_kept - head) >> 4, tail0 = head + (n16 << 4);
            if (threadIdx.x < head) dst[threadIdx.x] = s_bytes[threadIdx.x];
            const uint32_t sh = (head & 3u) * 8u;
            const uint32_t *s_words = reinterpret_cast<const uint32_t *>(s_bytes);
            for (uint32_t q = threadIdx.x; q < n16; q += TILE_THREADS) {
                const uint32_t w0 = (head + 16u * q) >> 2;                       // first aligned shared-memory word of this 16-byte piece
                const uint32_t a0 = s_words[w0], a1 = s_words[w0 + 1], a2 = s_words[w0 + 2], a3 = s_words[w0 + 3], a4 = s_words[w0 + 4];
                uint4 o;
                o.x = __funnelshift_r(a0, a1, sh); o.y = __funnelshift_r(a1, a2, sh);
                o.z = __funnelshift_r(a2, a3, sh); o.w = __funnelshift_r(a3, a4, sh);
                *reinterpret_cast<uint4 *>(dst + head + 16u * q) = o;
            }
            if (threadIdx.x < tile_kept - tail0) dst[tail0 + threadIdx.x] = s_bytes[tail0 + threadIdx.x];
        }
    }
}

struct Workspace { TileSummary *tiles; TileStart *starts; size_t bytes; };
static Workspace carve(void *ws, int64_t n_bytes) {
    const int64_t n_tiles = (n_bytes + TILE_BYTES - 1) / TILE_BYTES;
    Workspace w;
    unsigned char *base = static_cast<unsigned char *>(ws);
    const size_t a = ((size_t)n_tiles * sizeof(TileSummary) + 255) & ~(size_t)255;
    const size_t b = ((size_t)n_tiles * sizeof(TileStart) + 255) & ~(size_t)255;
    w.tiles = reinterpret_cast<TileSummary *>(base);
    w.starts = reinterpret_cast<TileStart *>(base ? base + a : nullptr);
    w.bytes = a + b + 256;
    return w;
}

}  // namespace fasta
}  // namespace phm

using namespace phm;

extern "C" size_t phm_fasta_workspace_bytes(int64_t n_bytes) {
    return fasta::carve(nullptr, n_bytes < 0 ? 0 : n_bytes).bytes;
}

extern "C" int phm_fasta_index(const uint8_t *d_raw, int64_t n_bytes, int64_t *d_result, void *d_workspace, size_t workspace_bytes,
                               void *stream) {
    PHM_REQUIRE(n_bytes >= 0, "n_bytes must be >= 0");
    PHM_REQUIRE(d_result != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_raw != nullptr || n_bytes == 0, "d_raw is null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_raw) & 15u) == 0, "d_raw must be 16-byte aligned");
    fasta::Workspace w = fasta::carve(d_workspace, n_bytes);
    if (workspace_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, w.bytes); return PHM_E_WORKSPACE; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n_tiles = (n_bytes + fasta::TILE_BYTES - 1) / fasta::TILE_BYTES;
    if (n_tiles > 0) {
        int64_t grid = (int64_t)sm_count() * 8;
        if (grid > n_tiles) grid = n_tiles;
        fasta::fasta_tile_kernel<<<(unsigned)grid, fasta::TILE_THREADS, 0, st>>>(d_raw, n_bytes, n_tiles, w.tiles);
        PHM_LAUNCH_CHECK();
    }
    fasta::fasta_chain_kernel<<<1, 1024, 0, st>>>(w.tiles, n_tiles, w.starts, d_result);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_fasta_extract(const uint8_t *d_raw, int64_t n_bytes, const int64_t *d_result, uint8_t *d_seq, int64_t *d_offsets,
                                 int64_t *d_header_pos, int64_t max_records, const void *d_workspace, size_t workspace_bytes,
                                 void *stream) {
    PHM_REQUIRE(n_bytes >= 0 && max_records >= 0, "negative size");
    PHM_REQUIRE(d_result != nullptr && d_workspace != nullptr && d_offsets != nullptr, "null pointer");
    PHM_REQUIRE((d_raw != nullptr && d_seq != nullptr) || n_bytes == 0, "d_raw / d_seq is null");
    PHM_REQUIRE(d_header_pos != nullptr || max_records == 0, "d_header_pos is null");
    fasta::Workspace w = fasta::carve(const_cast<void *>(d_workspace), n_bytes);
    if (workspace_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, w.bytes); return PHM_E_WORKSPACE; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n_tiles = (n_bytes + fasta::TILE_BYTES - 1) / fasta::TILE_BYTES;
    int64_t grid = (int64_t)sm_count() * 8;
    if (grid > n_tiles) grid = n_tiles;
    if (grid < 1) grid = 1;
    fasta::fasta_emit_kernel<<<(unsigned)grid, fasta::TILE_THREADS, 0, st>>>(d_raw, n_bytes, n_tiles, w.starts, d_result, d_seq, d_offsets,
                                                                             d_header_pos, max_records);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}
