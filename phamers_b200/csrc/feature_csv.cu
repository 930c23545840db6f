// Feature CSV text on the device (SURVEY.md 8(f): "fast writer needed at 1 M+ rows"): the k-mer count files of fileIO.save_counts /
// read_feature_file (reference scripts/fileIO.py:134-181): '#' header lines, then one row per contig, `id,c0,c1,...`.
//
// Format (int64 counts [n, F] + id bytes -> text), two calls:
//   csv_layout_kernel   one warp per row: the row's bytes = id length + max(F, 1) commas + sum of digits(v) + (v < 0) + 1 ('\n');
//                       each CTA scans its tile of ROW_TILE rows (tile-local offsets + the tile's total)
//   csv_chain_kernel    one CTA: exclusive scan of the tile totals (the text size lands in the workspace)
//   csv_offsets_kernel  tile base + local offset -> row offsets [n + 1]
//   csv_format_kernel   one warp per row: the id, then 32 fields at a time -- a warp scan of the field lengths places each lane's
//                       field, which it converts two digits per step from a 200-byte table -- into a per-warp staging buffer in
//                       shared memory that mirrors the 16-byte alignment of the text, flushed as whole 16-byte words (rows longer
//                       than the buffer go out in pieces; only the partial words at a row's two ends are written byte by byte)
//
// Parse (text -> int64 counts [rows, F] + id byte ranges), the same grammar as fileIO.read_feature_file on the files it accepts:
//   bytes: printable ASCII, TAB, CR and LF only (any other byte: decline); lines end at LF or CR (universal newlines: the empty line
//   inside a CRLF is skipped like any blank line); a line is cut at its first '#' and stripped of blanks (space, TAB); an empty result
//   is skipped; a data line is `id,field,...`: the id is everything before the first ',' (its inner and trailing blanks kept), and
//   each field is [ \t]*[+-]?[0-9]{1,18}[ \t]* (18 digits always fit int64).  Every data line has the same number of fields.
//   Anything else declines the whole file (the host road then runs, and returns or raises what it always did).
//   csv_lines_kernel    per 4 KB tile: its line starts (the first byte of the file, and every byte after an LF or CR)
//   csv_chain_kernel    line number of each tile's first line start
//   csv_index_kernel    per tile: bytes outside the alphabet; the line starts compacted in shared memory, then one warp per line
//                       (reading past the tile as far as the line goes) finds the cut, the first non-blank byte, the commas, and
//                       checks every field; per tile its data lines, per CTA the field-count range, the first data line and the first
//                       decline (line << 3 | reason)
//   csv_chain_kernel    row index of each tile's first data line
//   csv_index_kernel<LOCATE>  only when the field counts differ: the first data line whose count is not the first data line's
//   csv_result_kernel   the result block
//   csv_fill_kernel     per tile again: which lines are data lines (one warp each), their ranks in the tile, then one warp per data
//                       line parses its fields into its row and records the id's byte range
// Every read is bounded by the text (whose allocation is readable up to the next multiple of 16 bytes, as for phm_fasta_index) and
// every write by the outputs, whatever the bytes; malformed text ends in a decline, never a trap.
#include "byte_class.cuh"
#include "phm_common.cuh"

namespace phm {
namespace csv {

// ================================================ shared ================================================
// exclusive scan of int64 values in place (one CTA, each thread a contiguous range); the sum goes to *total
__global__ void __launch_bounds__(1024) csv_chain_kernel(int64_t *__restrict__ vals, int64_t n, int64_t *__restrict__ total) {
    __shared__ int64_t s_warp[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t per = (n + 1023) / 1024;
    const int64_t lo = (int64_t)threadIdx.x * per < n ? (int64_t)threadIdx.x * per : n;
    const int64_t hi = lo + per < n ? lo + per : n;
    int64_t sum = 0;
    for (int64_t i = lo; i < hi; ++i) sum += vals[i];
    int64_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int64_t base = incl - sum;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    for (int64_t i = lo; i < hi; ++i) {
        const int64_t x = vals[i];
        vals[i] = base;
        base += x;
    }
    if (threadIdx.x == 1023) *total = base;
}

__device__ __forceinline__ uint32_t eq16(const uint32_t w[4], uint32_t pattern) {     // bytes equal to `pattern`'s byte
    uint32_t m = 0u;
#pragma unroll
    for (int q = 0; q < 4; ++q) m |= gather4(zero_bytes(w[q] ^ pattern)) << (4 * q);
    return m;
}
__device__ __forceinline__ uint32_t valid16(int64_t p0, int64_t n) {                  // bytes of [p0, p0 + 16) before n
    return p0 >= n ? 0u : (p0 + 16 <= n ? 0xFFFFu : (1u << (int)(n - p0)) - 1u);
}

// ================================================ format ================================================
constexpr int FMT_WARPS = 8;
constexpr int FMT_THREADS = FMT_WARPS * 32;
constexpr int ROW_TILE = FMT_THREADS;                  // rows per layout tile (one per thread in the tile's scan)
constexpr int STAGE = 2048;                            // staging bytes per warp
constexpr int CHUNK_MAX = 32 * 21;                     // 32 fields of ',' '-' and 19 digits

__device__ __forceinline__ uint64_t magnitude(int64_t v) { return v < 0 ? 0ull - (uint64_t)v : (uint64_t)v; }
__device__ __forceinline__ int n_digits(uint64_t u) {
    int d = 1;
    for (uint64_t t = 10u; d < 19 && u >= t; t *= 10u) ++d;
    return d;
}
__device__ __forceinline__ int field_bytes(int64_t v) { return 1 + (v < 0 ? 1 : 0) + n_digits(magnitude(v)); }
// the id bytes of row r, clamped to [0, id_bytes) and to a non-negative length
__device__ __forceinline__ void id_range(const int64_t *id_off, int64_t r, int64_t id_bytes, int64_t &lo, int64_t &hi) {
    lo = id_off[r];
    hi = id_off[r + 1];
    lo = lo < 0 ? 0 : (lo > id_bytes ? id_bytes : lo);
    hi = hi < lo ? lo : (hi > id_bytes ? id_bytes : hi);
}

__global__ void __launch_bounds__(FMT_THREADS) csv_layout_kernel(const int64_t *__restrict__ counts, int64_t n_rows, int64_t n_cols,
                                                                 const int64_t *__restrict__ id_off, int64_t id_bytes,
                                                                 int64_t *__restrict__ row_off, int64_t *__restrict__ tile_sums,
                                                                 int64_t n_tiles) {
    __shared__ int64_t s_len[ROW_TILE];
    __shared__ int64_t s_warp[FMT_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t r0 = tile * ROW_TILE;
        for (int i = warp; i < ROW_TILE; i += FMT_WARPS) {
            const int64_t r = r0 + i;
            int64_t len = 0;
            if (r < n_rows) {
                const int64_t *row = counts + r * n_cols;
                for (int64_t c = lane; c < n_cols; c += 32) len += field_bytes(row[c]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) len += __shfl_xor_sync(FULL, len, o);
                int64_t lo, hi;
                id_range(id_off, r, id_bytes, lo, hi);
                len += (hi - lo) + (n_cols == 0 ? 1 : 0) + 1;
            }
            if (lane == 0) s_len[i] = len;
        }
        __syncthreads();
        const int64_t v = s_len[threadIdx.x];
        int64_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int64_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < FMT_WARPS; ++w) {
            before += w < warp ? s_warp[w] : 0;
            total += s_warp[w];
        }
        if (r0 + threadIdx.x < n_rows) row_off[r0 + threadIdx.x] = before + incl - v;
        if (threadIdx.x == 0) tile_sums[tile] = total;
        __syncthreads();                                           // s_len / s_warp are rewritten by the next tile
    }
}

__global__ void csv_offsets_kernel(int64_t *__restrict__ row_off, int64_t n_rows, const int64_t *__restrict__ tile_base,
                                   const int64_t *__restrict__ total) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += (int64_t)gridDim.x * blockDim.x)
        row_off[r] = r < n_rows ? row_off[r] + tile_base[r / ROW_TILE] : *total;
}

// Staged bytes s[lo, end) go to text[abase + lo, abase + end), abase a multiple of 16: whole words as 16-byte stores, the partial words
// at either end byte by byte.  Not final: end = cur rounded down to 16, and the rest of the last word moves to the front.
__device__ __forceinline__ void flush(uint8_t *s, int &lo, int &cur, int64_t &abase, bool final, uint8_t *text, int64_t text_bytes,
                                      int lane) {
    __syncwarp();
    const int end = final ? cur : (cur & ~15);
    const int w_lo = (lo + 15) >> 4, w_hi = end >> 4;
    const int head_end = (w_lo << 4) < end ? (w_lo << 4) : end;
    for (int j = lo + lane; j < head_end; j += 32) {
        const int64_t g = abase + j;
        if (g >= 0 && g < text_bytes) text[g] = s[j];
    }
    for (int q = w_lo + lane; q < w_hi; q += 32) {
        const int64_t g = abase + 16 * (int64_t)q;
        if (g >= 0 && g + 16 <= text_bytes) {
            *reinterpret_cast<uint4 *>(text + g) = *reinterpret_cast<const uint4 *>(s + 16 * q);
        } else {
            for (int j = 0; j < 16; ++j)
                if (g + j >= 0 && g + j < text_bytes) text[g + j] = s[16 * q + j];
        }
    }
    for (int j = ((w_hi > w_lo ? w_hi : w_lo) << 4) + lane; j < end; j += 32) {
        const int64_t g = abase + j;
        if (g >= 0 && g < text_bytes) text[g] = s[j];
    }
    __syncwarp();
    if (!final) {
        const int rest = cur - end;                                    // < 16
        const uint8_t b = lane < rest ? s[end + lane] : 0;
        __syncwarp();
        if (lane < rest) s[lane] = b;
        abase += end;
        cur = rest;
        lo = 0;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(FMT_THREADS) csv_format_kernel(const int64_t *__restrict__ counts, int64_t n_rows, int64_t n_cols,
                                                                 const uint8_t *__restrict__ ids, const int64_t *__restrict__ id_off,
                                                                 int64_t id_bytes, const int64_t *__restrict__ row_off,
                                                                 uint8_t *__restrict__ text, int64_t text_bytes) {
    __shared__ __align__(16) uint8_t s_stage[FMT_WARPS][STAGE];
    __shared__ uint8_t s_pairs[200];                                   // "00" "01" ... "99"
    for (int i = threadIdx.x; i < 200; i += blockDim.x) s_pairs[i] = (uint8_t)('0' + ((i & 1) ? (i >> 1) % 10 : (i >> 1) / 10));
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *s = s_stage[warp];
    for (int64_t r = (int64_t)blockIdx.x * FMT_WARPS + warp; r < n_rows; r += (int64_t)gridDim.x * FMT_WARPS) {
        const int64_t off = row_off[r];
        int64_t abase = off & ~(int64_t)15;
        int lo = (int)(off - abase), cur = lo;
        int64_t a, b;
        id_range(id_off, r, id_bytes, a, b);
        for (int64_t p = a; p < b; p += 512) {
            const int m = b - p < 512 ? (int)(b - p) : 512;
            if (cur + m > STAGE) flush(s, lo, cur, abase, false, text, text_bytes, lane);
            for (int j = lane; j < m; j += 32) s[cur + j] = ids[p + j];
            cur += m;
        }
        if (n_cols == 0) {                                              // no fields: 'id,'
            if (cur + 1 > STAGE) flush(s, lo, cur, abase, false, text, text_bytes, lane);
            if (lane == 0) s[cur] = ',';
            cur += 1;
        }
        const int64_t *row = counts + r * n_cols;
        for (int64_t c0 = 0; c0 < n_cols; c0 += 32) {
            if (cur + CHUNK_MAX > STAGE) flush(s, lo, cur, abase, false, text, text_bytes, lane);
            const int64_t c = c0 + lane;
            const int64_t v = c < n_cols ? row[c] : 0;
            const int len = c < n_cols ? field_bytes(v) : 0;
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += up;
            }
            if (len) {
                uint8_t *p = s + cur + incl - len;
                *p++ = ',';
                if (v < 0) *p++ = '-';
                uint8_t *e = s + cur + incl;
                uint64_t u = magnitude(v);
                while (u >= 100u) {
                    const uint64_t q = u / 100u;
                    const uint32_t two = (uint32_t)(u - q * 100u) * 2u;
                    e -= 2;
                    e[0] = s_pairs[two];
                    e[1] = s_pairs[two + 1];
                    u = q;
                }
                if (u >= 10u) {
                    e[-2] = s_pairs[2u * (uint32_t)u];
                    e[-1] = s_pairs[2u * (uint32_t)u + 1u];
                } else {
                    e[-1] = (uint8_t)('0' + (uint32_t)u);
                }
            }
            cur += __shfl_sync(FULL, incl, 31);
        }
        if (cur + 1 > STAGE) flush(s, lo, cur, abase, false, text, text_bytes, lane);
        if (lane == 0) s[cur] = '\n';
        cur += 1;
        flush(s, lo, cur, abase, true, text, text_bytes, lane);
    }
}

struct FormatWorkspace { int64_t *tile_sums; int64_t *total; size_t bytes; };
static FormatWorkspace carve_format(void *ws, int64_t n_rows) {
    const int64_t n_tiles = (n_rows + ROW_TILE - 1) / ROW_TILE;
    FormatWorkspace w;
    unsigned char *base = static_cast<unsigned char *>(ws);
    const size_t a = ((size_t)(n_tiles + 1) * sizeof(int64_t) + 255) & ~(size_t)255;
    w.tile_sums = reinterpret_cast<int64_t *>(base);
    w.total = reinterpret_cast<int64_t *>(base ? base + a : nullptr);
    w.bytes = a + 256;
    return w;
}

// ================================================ parse ================================================
constexpr int PT_WARPS = 8;
constexpr int PT_THREADS = PT_WARPS * 32;
constexpr int PT_TILE = PT_THREADS * 16;                // 4 KB: at most 4 096 line starts, kept as 16-bit offsets in shared memory
constexpr uint64_t WIDE = 0xFFFFFFu;                    // field counts are compared up to 2^24 - 1 when the first data line is located
enum { ACC_FMIN, ACC_FMAX, ACC_KEY, ACC_FIRST, ACC_ROWS, ACC_LINES, ACC_N };

__device__ __forceinline__ void load16(const uint8_t *text, int64_t n, int64_t p0, uint32_t w[4]) {
    w[0] = w[1] = w[2] = w[3] = 0x0A0A0A0Au;
    if (p0 < n) {
        const uint4 v = *reinterpret_cast<const uint4 *>(text + p0);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    }
}
// line starts among the 16 bytes at p0 (16-aligned): the file's first byte and every byte after an LF or CR, before n
__device__ __forceinline__ uint32_t line_starts16(const uint8_t *text, int64_t n, int64_t p0, const uint32_t w[4]) {
    const uint32_t valid = valid16(p0, n);
    if (!valid) return 0u;
    const uint32_t nl = eq16(w, 0x0A0A0A0Au) | eq16(w, 0x0D0D0D0Du);
    const uint32_t prev = p0 == 0 ? 10u : text[p0 - 1];
    return ((nl << 1) | ((prev == 10u || prev == 13u) ? 1u : 0u)) & valid;
}

// [a, b): [ \t]*[+-]?[0-9]{1,18}[ \t]*
__device__ __forceinline__ bool parse_field(const uint8_t *t, int64_t a, int64_t b, int64_t &out) {
    int64_t i = a;
    while (i < b && (t[i] == ' ' || t[i] == '\t')) ++i;
    bool neg = false;
    if (i < b && (t[i] == '+' || t[i] == '-')) { neg = t[i] == '-'; ++i; }
    const int64_t d0 = i;
    uint64_t v = 0u;
    while (i < b && (uint32_t)(t[i] - '0') < 10u) { v = v * 10u + (uint32_t)(t[i] - '0'); ++i; }
    const int64_t nd = i - d0;
    while (i < b && (t[i] == ' ' || t[i] == '\t')) ++i;
    out = neg ? (int64_t)(0ull - v) : (int64_t)v;
    return nd >= 1 && nd <= 18 && i == b;
}

enum { SCAN_DATA, SCAN_CHECK, SCAN_FILL };
struct LineInfo { int64_t id_lo, id_hi, fields; int status; bool data; };

// One warp reads the line that starts at s, 512 bytes per step, up to its cut (the first LF, CR or '#', or n).  SCAN_DATA stops once it
// is known whether the line holds a non-blank byte; SCAN_CHECK counts the fields and checks each; SCAN_FILL also writes field j to
// out[j] for j < n_cols.  A field is parsed by the lane holding the comma that ends it; the last field by lane 0.  Warp-uniform result.
template <int MODE>
__device__ __forceinline__ LineInfo scan_line(const uint8_t *__restrict__ text, int64_t n, int64_t s, int64_t *__restrict__ out, int64_t n_cols,
                              int lane) {
    int64_t first_nb = -1, first_comma = -1, prev_comma = -1, n_comma = 0, cut = n;
    bool bad = false;
    for (int64_t base = s & ~(int64_t)15;; base += 512) {
        const int64_t p0 = base + 16 * lane;
        uint32_t w[4];
        load16(text, n, p0, w);
        const uint32_t from_s = p0 >= s ? 0xFFFFu : (p0 + 16 <= s ? 0u : (0xFFFFu << (int)(s - p0)) & 0xFFFFu);
        const uint32_t term = ((eq16(w, 0x0A0A0A0Au) | eq16(w, 0x0D0D0D0Du) | eq16(w, 0x23232323u) | (~valid16(p0, n) & 0xFFFFu))) & from_s;
        const uint32_t t_lanes = __ballot_sync(FULL, term != 0u);
        const int cut_lane = t_lanes ? __ffs(t_lanes) - 1 : 32;
        const uint32_t live = lane < cut_lane ? from_s : (lane == cut_lane ? from_s & ((1u << (__ffs(term) - 1)) - 1u) : 0u);
        if (first_nb < 0) {
            const uint32_t nb = live & ~(eq16(w, 0x20202020u) | eq16(w, 0x09090909u));
            const uint32_t nb_lanes = __ballot_sync(FULL, nb != 0u);
            if (nb_lanes) {
                const int l = __ffs(nb_lanes) - 1;
                first_nb = __shfl_sync(FULL, p0 + (nb ? __ffs(nb) - 1 : 0), l);
            }
        }
        if (cut_lane < 32) cut = __shfl_sync(FULL, p0 + (term ? __ffs(term) - 1 : 0), cut_lane);
        if (MODE == SCAN_DATA && (first_nb >= 0 || cut_lane < 32)) break;
        const uint32_t cm = live & eq16(w, 0x2C2C2C2Cu);
        const int cnt = __popc(cm);
        int incl = cnt;
        int64_t last = cm ? p0 + 31 - __clz(cm) : -1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, incl, o);
            const int64_t up_last = __shfl_up_sync(FULL, last, o);
            if (lane >= o) { incl += up; last = up_last > last ? up_last : last; }
        }
        int64_t prev = __shfl_up_sync(FULL, last, 1);
        if (lane == 0) prev = -1;
        prev = prev > prev_comma ? prev : prev_comma;
        int64_t rank = n_comma + incl - cnt;
        for (uint32_t m = cm; m; m &= m - 1u, ++rank) {
            const int64_t pos = p0 + __ffs(m) - 1;
            if (rank > 0) {
                int64_t v;
                bad |= !parse_field(text, prev + 1, pos, v);
                if (MODE == SCAN_FILL && rank - 1 < n_cols) out[rank - 1] = v;
            }
            prev = pos;
        }
        const uint32_t c_lanes = __ballot_sync(FULL, cm != 0u);
        if (first_comma < 0 && c_lanes) first_comma = __shfl_sync(FULL, p0 + (cm ? __ffs(cm) - 1 : 0), __ffs(c_lanes) - 1);
        n_comma += __shfl_sync(FULL, incl, 31);
        const int64_t l31 = __shfl_sync(FULL, last, 31);
        prev_comma = l31 > prev_comma ? l31 : prev_comma;
        if (cut_lane < 32) break;
    }
    LineInfo L;
    L.data = first_nb >= 0;
    L.fields = n_comma;
    L.id_lo = first_nb;
    L.id_hi = first_comma;
    if (MODE != SCAN_DATA && L.data && n_comma > 0 && lane == 0) {
        int64_t v;
        bad |= !parse_field(text, prev_comma + 1, cut, v);
        if (MODE == SCAN_FILL && n_comma - 1 < n_cols) out[n_comma - 1] = v;
    }
    bad = __any_sync(FULL, bad);
    L.status = !L.data ? PHM_CSV_OK : (n_comma == 0 ? PHM_CSV_NO_COMMA : (bad ? PHM_CSV_FIELD : PHM_CSV_OK));
    return L;
}

// the tile's line starts as 16-bit offsets in s_ls, in file order; returns their number.  Also the thread's 16 bytes and line starts.
__device__ __forceinline__ int tile_line_starts(const uint8_t *text, int64_t n, int64_t t0, uint16_t *s_ls, uint32_t *s_warp,
                                                uint32_t w[4], uint32_t &ls, uint32_t &before) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t p0 = t0 + 16 * threadIdx.x;
    load16(text, n, p0, w);
    ls = line_starts16(text, n, p0, w);
    const uint32_t cnt = __popc(ls);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    __syncthreads();                                               // the previous tile is done with s_ls / s_warp
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t total = 0u;
    before = incl - cnt;
#pragma unroll
    for (int i = 0; i < PT_WARPS; ++i) {
        before += i < warp ? s_warp[i] : 0u;
        total += s_warp[i];
    }
    uint32_t k = before;
    for (uint32_t m = ls; m; m &= m - 1u) s_ls[k++] = (uint16_t)(16 * threadIdx.x + __ffs(m) - 1);
    __syncthreads();
    return (int)total;
}

__device__ __forceinline__ unsigned long long umin(unsigned long long a, unsigned long long b) { return a < b ? a : b; }
__device__ __forceinline__ unsigned long long umax(unsigned long long a, unsigned long long b) { return a > b ? a : b; }

__global__ void __launch_bounds__(PT_THREADS) csv_lines_kernel(const uint8_t *__restrict__ text, int64_t n, int64_t n_tiles,
                                                               int64_t *__restrict__ tile_lines, unsigned long long *__restrict__ acc) {
    __shared__ uint32_t s_warp[PT_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        acc[ACC_FMIN] = ~0ull; acc[ACC_FMAX] = 0ull; acc[ACC_KEY] = ~0ull; acc[ACC_FIRST] = ~0ull; acc[ACC_ROWS] = 0ull;
        acc[ACC_LINES] = 0ull;
    }
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t p0 = tile * PT_TILE + 16 * threadIdx.x;
        uint32_t w[4];
        load16(text, n, p0, w);
        uint32_t c = __popc(line_starts16(text, n, p0, w));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
        __syncthreads();
        if (lane == 0) s_warp[warp] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int64_t t = 0;
            for (int i = 0; i < PT_WARPS; ++i) t += s_warp[i];
            tile_lines[tile] = t;
        }
    }
}

template <bool LOCATE>
__global__ void __launch_bounds__(PT_THREADS) csv_index_kernel(const uint8_t *__restrict__ text, int64_t n, int64_t n_tiles,
                                                               const int64_t *__restrict__ line_base, int64_t *__restrict__ tile_rows,
                                                               unsigned long long *__restrict__ acc) {
    __shared__ uint16_t s_ls[PT_TILE];
    __shared__ uint32_t s_warp[PT_WARPS];
    __shared__ uint32_t s_rows;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t f0 = 0u;
    if (LOCATE) {                                                  // only when the data lines' field counts differ
        if (acc[ACC_FMAX] == 0ull || acc[ACC_FMIN] == acc[ACC_FMAX]) return;
        f0 = acc[ACC_FIRST] & WIDE;
    }
    unsigned long long fmin = ~0ull, fmax = 0ull, key = ~0ull, first = ~0ull;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t t0 = tile * PT_TILE;
        uint32_t w[4], ls, before;
        const int lines = tile_line_starts(text, n, t0, s_ls, s_warp, w, ls, before);
        const int64_t lb = line_base[tile];
        if (!LOCATE) {
            // bytes outside printable ASCII + TAB, CR, LF; the line of the first one = line starts up to and including it
            uint32_t ctrl = 0u, high = 0u;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                ctrl |= gather4(zero_bytes(w[q] & 0xE0E0E0E0u)) << (4 * q);
                high |= (gather4(w[q] & 0x80808080u) | gather4(zero_bytes(w[q] ^ 0x7F7F7F7Fu))) << (4 * q);
            }
            const uint32_t odd = ((ctrl & ~(eq16(w, 0x09090909u) | eq16(w, 0x0A0A0A0Au) | eq16(w, 0x0D0D0D0Du))) | high) &
                                 valid16(t0 + 16 * threadIdx.x, n);
            if (odd) {
                const int j = __ffs(odd) - 1;
                const unsigned long long line = (unsigned long long)(lb + before + __popc(ls & ((2u << j) - 1u)));
                key = umin(key, (line << 3) | PHM_CSV_BYTE);
            }
            if (threadIdx.x == 0) s_rows = 0u;
            __syncthreads();
        }
        for (int k = warp; k < lines; k += PT_WARPS) {
            const LineInfo L = scan_line<SCAN_CHECK>(text, n, t0 + s_ls[k], nullptr, 0, lane);
            if (lane == 0 && L.data) {
                const unsigned long long line = (unsigned long long)(lb + k + 1), f = (unsigned long long)L.fields;
                const unsigned long long fw = f < WIDE ? f : WIDE;
                if (LOCATE) {
                    if (fw != f0) key = umin(key, (line << 3) | PHM_CSV_RAGGED);
                } else {
                    atomicAdd(&s_rows, 1u);
                    fmin = umin(fmin, f);
                    fmax = umax(fmax, f);
                    first = umin(first, (line << 24) | fw);
                    if (L.status != PHM_CSV_OK) key = umin(key, (line << 3) | (unsigned long long)L.status);
                }
            }
        }
        if (!LOCATE) {
            __syncthreads();
            if (threadIdx.x == 0) tile_rows[tile] = s_rows;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        fmin = umin(fmin, __shfl_xor_sync(FULL, fmin, o));
        fmax = umax(fmax, __shfl_xor_sync(FULL, fmax, o));
        key = umin(key, __shfl_xor_sync(FULL, key, o));
        first = umin(first, __shfl_xor_sync(FULL, first, o));
    }
    if (lane == 0) {
        if (key != ~0ull) atomicMin(&acc[ACC_KEY], key);
        if (!LOCATE && fmax != 0ull) {
            atomicMin(&acc[ACC_FMIN], fmin);
            atomicMax(&acc[ACC_FMAX], fmax);
            atomicMin(&acc[ACC_FIRST], first);
        }
    }
}

// result[0] data rows, [1] fields, [2] PHM_CSV_* reason (0: accepted), [3] line of the first decline (1-based; 0 when accepted)
__global__ void csv_result_kernel(const unsigned long long *__restrict__ acc, const int64_t *__restrict__ rows, int64_t *__restrict__ result) {
    const unsigned long long key = acc[ACC_KEY];
    const int64_t r = *rows;
    int64_t reason = PHM_CSV_OK, line = 0;
    if (key != ~0ull) {
        reason = (int64_t)(key & 7u);
        line = (int64_t)(key >> 3);
    } else if (r > 0 && acc[ACC_FMIN] != acc[ACC_FMAX]) {          // widths past 2^24 - 1 that differ: reported at the first data line
        reason = PHM_CSV_RAGGED;
        line = (int64_t)(acc[ACC_FIRST] >> 24);
    }
    result[0] = r;
    result[1] = r > 0 ? (int64_t)acc[ACC_FMIN] : 0;
    result[2] = reason;
    result[3] = line;
}

__global__ void __launch_bounds__(PT_THREADS, 4) csv_fill_kernel(const uint8_t *__restrict__ text, int64_t n, int64_t n_tiles,
                                                              const int64_t *__restrict__ row_base, int64_t *__restrict__ counts,
                                                              int64_t *__restrict__ id_ranges, int64_t max_rows, int64_t n_cols) {
    __shared__ uint16_t s_ls[PT_TILE];
    __shared__ uint16_t s_rank[PT_TILE];                           // bit 15: data line; bits 0-14: data lines before it in the tile
    __shared__ uint32_t s_warp[PT_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int PER = PT_TILE / PT_THREADS;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t t0 = tile * PT_TILE;
        uint32_t w[4], ls, before;
        const int lines = tile_line_starts(text, n, t0, s_ls, s_warp, w, ls, before);
        for (int k = warp; k < lines; k += PT_WARPS) {
            const LineInfo L = scan_line<SCAN_DATA>(text, n, t0 + s_ls[k], nullptr, 0, lane);
            if (lane == 0) s_rank[k] = L.data ? 1u : 0u;
        }
        __syncthreads();
        uint32_t mine = 0u;
        for (int j = 0; j < PER; ++j) {
            const int k = PER * threadIdx.x + j;
            mine += k < lines ? s_rank[k] : 0u;
        }
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        __syncthreads();
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t rank = incl - mine;
        for (int i = 0; i < warp; ++i) rank += s_warp[i];
        for (int j = 0; j < PER; ++j) {
            const int k = PER * threadIdx.x + j;
            if (k < lines) {
                const uint32_t d = s_rank[k];
                s_rank[k] = (uint16_t)((d << 15) | rank);
                rank += d;
            }
        }
        __syncthreads();
        const int64_t rb = row_base[tile];
        for (int k = warp; k < lines; k += PT_WARPS) {
            const uint32_t e = s_rank[k];
            const int64_t row = rb + (e & 0x7FFFu);
            if (!(e >> 15) || row >= max_rows) continue;
            const LineInfo L = scan_line<SCAN_FILL>(text, n, t0 + s_ls[k], counts + row * n_cols, n_cols, lane);
            if (lane == 0) { id_ranges[2 * row] = L.id_lo; id_ranges[2 * row + 1] = L.id_hi; }
        }
    }
}

struct ParseWorkspace { int64_t *tile_lines; int64_t *tile_rows; unsigned long long *acc; size_t bytes; };
static ParseWorkspace carve_parse(void *ws, int64_t n_bytes) {
    const int64_t n_tiles = (n_bytes + PT_TILE - 1) / PT_TILE;
    ParseWorkspace w;
    unsigned char *base = static_cast<unsigned char *>(ws);
    const size_t a = ((size_t)(n_tiles + 1) * sizeof(int64_t) + 255) & ~(size_t)255;
    w.tile_lines = reinterpret_cast<int64_t *>(base);
    w.tile_rows = reinterpret_cast<int64_t *>(base ? base + a : nullptr);
    w.acc = reinterpret_cast<unsigned long long *>(base ? base + 2 * a : nullptr);
    w.bytes = 2 * a + 256;
    return w;
}

static int64_t grid_for(int64_t items) {
    int64_t grid = (int64_t)sm_count() * 8;
    if (grid > items) grid = items;
    return grid < 1 ? 1 : grid;
}

}  // namespace csv
}  // namespace phm

using namespace phm;

extern "C" size_t phm_counts_csv_workspace_bytes(int64_t n_rows) {
    return csv::carve_format(nullptr, n_rows < 0 ? 0 : n_rows).bytes;
}

extern "C" int phm_counts_csv_layout(const int64_t *d_counts, int64_t n_rows, int64_t n_cols, const int64_t *d_id_offsets,
                                     int64_t id_bytes, int64_t *d_row_offsets, void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(n_rows >= 0 && n_cols >= 0 && id_bytes >= 0, "negative size");
    PHM_REQUIRE(d_id_offsets != nullptr && d_row_offsets != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_counts != nullptr || n_rows == 0 || n_cols == 0, "d_counts is null");
    csv::FormatWorkspace w = csv::carve_format(d_workspace, n_rows);
    if (workspace_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, w.bytes); return PHM_E_WORKSPACE; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n_tiles = (n_rows + csv::ROW_TILE - 1) / csv::ROW_TILE;
    if (n_tiles > 0) {
        csv::csv_layout_kernel<<<(unsigned)csv::grid_for(n_tiles), csv::FMT_THREADS, 0, st>>>(d_counts, n_rows, n_cols, d_id_offsets,
                                                                                             id_bytes, d_row_offsets, w.tile_sums, n_tiles);
        PHM_LAUNCH_CHECK();
    }
    csv::csv_chain_kernel<<<1, 1024, 0, st>>>(w.tile_sums, n_tiles, w.total);
    PHM_LAUNCH_CHECK();
    csv::csv_offsets_kernel<<<(unsigned)csv::grid_for((n_rows + 256) / 256), 256, 0, st>>>(d_row_offsets, n_rows, w.tile_sums, w.total);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_counts_csv_format(const int64_t *d_counts, int64_t n_rows, int64_t n_cols, const uint8_t *d_ids,
                                     const int64_t *d_id_offsets, int64_t id_bytes, const int64_t *d_row_offsets, uint8_t *d_text,
                                     int64_t text_bytes, void *stream) {
    PHM_REQUIRE(n_rows >= 0 && n_cols >= 0 && id_bytes >= 0 && text_bytes >= 0, "negative size");
    PHM_REQUIRE(d_id_offsets != nullptr && d_row_offsets != nullptr, "null pointer");
    PHM_REQUIRE(d_counts != nullptr || n_rows == 0 || n_cols == 0, "d_counts is null");
    PHM_REQUIRE(d_ids != nullptr || id_bytes == 0, "d_ids is null");
    PHM_REQUIRE(d_text != nullptr || text_bytes == 0, "d_text is null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15u) == 0, "d_text must be 16-byte aligned");
    if (n_rows == 0) return PHM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    csv::csv_format_kernel<<<(unsigned)csv::grid_for((n_rows + csv::FMT_WARPS - 1) / csv::FMT_WARPS), csv::FMT_THREADS, 0, st>>>(
        d_counts, n_rows, n_cols, d_ids, d_id_offsets, id_bytes, d_row_offsets, d_text, text_bytes);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" size_t phm_feature_csv_workspace_bytes(int64_t n_bytes) {
    return csv::carve_parse(nullptr, n_bytes < 0 ? 0 : n_bytes).bytes;
}

extern "C" int phm_feature_csv_index(const uint8_t *d_text, int64_t n_bytes, int64_t *d_result, void *d_workspace,
                                     size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(n_bytes >= 0 && n_bytes < ((int64_t)1 << 40), "n_bytes must be in [0, 2^40)");
    PHM_REQUIRE(d_result != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_text != nullptr || n_bytes == 0, "d_text is null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15u) == 0, "d_text must be 16-byte aligned");
    csv::ParseWorkspace w = csv::carve_parse(d_workspace, n_bytes);
    if (workspace_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, w.bytes); return PHM_E_WORKSPACE; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n_tiles = (n_bytes + csv::PT_TILE - 1) / csv::PT_TILE;
    int64_t *lines_total = reinterpret_cast<int64_t *>(w.acc + csv::ACC_LINES);
    int64_t *rows_total = reinterpret_cast<int64_t *>(w.acc + csv::ACC_ROWS);
    const unsigned grid = (unsigned)csv::grid_for(n_tiles);
    csv::csv_lines_kernel<<<grid, csv::PT_THREADS, 0, st>>>(d_text, n_bytes, n_tiles, w.tile_lines, w.acc);
    PHM_LAUNCH_CHECK();
    csv::csv_chain_kernel<<<1, 1024, 0, st>>>(w.tile_lines, n_tiles, lines_total);
    PHM_LAUNCH_CHECK();
    csv::csv_index_kernel<false><<<grid, csv::PT_THREADS, 0, st>>>(d_text, n_bytes, n_tiles, w.tile_lines, w.tile_rows, w.acc);
    PHM_LAUNCH_CHECK();
    csv::csv_chain_kernel<<<1, 1024, 0, st>>>(w.tile_rows, n_tiles, rows_total);
    PHM_LAUNCH_CHECK();
    csv::csv_index_kernel<true><<<grid, csv::PT_THREADS, 0, st>>>(d_text, n_bytes, n_tiles, w.tile_lines, w.tile_rows, w.acc);
    PHM_LAUNCH_CHECK();
    csv::csv_result_kernel<<<1, 1, 0, st>>>(w.acc, rows_total, d_result);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_feature_csv_parse(const uint8_t *d_text, int64_t n_bytes, int64_t *d_counts, int64_t *d_id_ranges, int64_t max_rows,
                                     int64_t n_cols, const void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(n_bytes >= 0 && n_bytes < ((int64_t)1 << 40), "n_bytes must be in [0, 2^40)");
    PHM_REQUIRE(max_rows >= 0 && n_cols >= 0, "negative size");
    PHM_REQUIRE(d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(d_text != nullptr || n_bytes == 0, "d_text is null");
    PHM_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15u) == 0, "d_text must be 16-byte aligned");
    PHM_REQUIRE(max_rows == 0 || (d_id_ranges != nullptr && (d_counts != nullptr || n_cols == 0)), "d_counts / d_id_ranges is null");
    csv::ParseWorkspace w = csv::carve_parse(const_cast<void *>(d_workspace), n_bytes);
    if (workspace_bytes < w.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, w.bytes); return PHM_E_WORKSPACE; }
    const int64_t n_tiles = (n_bytes + csv::PT_TILE - 1) / csv::PT_TILE;
    if (n_tiles == 0 || max_rows == 0) return PHM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    csv::csv_fill_kernel<<<(unsigned)csv::grid_for(n_tiles), csv::PT_THREADS, 0, st>>>(d_text, n_bytes, n_tiles, w.tile_rows, d_counts,
                                                                                       d_id_ranges, max_rows, n_cols);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}
