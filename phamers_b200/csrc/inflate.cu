// BGZF decompression on the device: every member of a BGZF file (the blocked gzip of bgzip / htslib) is an independent raw
// DEFLATE stream (RFC 1951) of at most 64 KiB of output, and the host finds every member and its output offset from the headers
// alone (fileIO.bgzf_members), so thousands of members decode at once.  phm_inflate writes member i's output to
// d_out[out_offset, out_offset + isize) and checks its CRC32 and length against the gzip trailer, as gzip does.
//
// Layout: one warp per member (grid-stride over the table).  All 32 lanes run the same Huffman decode on the same 64-bit bit
// buffer (the decode tables are in the warp's shared memory, so every table read is a broadcast), which keeps the warp converged
// without a shuffle per symbol; lane 0 stores literals, and the whole warp copies matches and stored blocks.  A back-reference
// never leaves its member, so it reads output this warp has just written (__syncwarp orders those accesses).
//
// Decode tables (RFC 1951 canonical codes): a primary table indexed by the next LIT_BITS / DIST_BITS / CL_BITS input bits gives
// (symbol, length) for every code no longer than that; a longer code (rare: lit/len codes of 11..15 bits, distance codes of
// 9..15) is decoded bit by bit from the per-length counts and the symbols sorted by code (the method of zlib's puff.c).
// The code-length code has at most 7 bits and is always decoded from its primary table.
//
// What is accepted is what zlib accepts: an over-subscribed code is an error; an incomplete code only when it is a single code of
// one bit in a lit/len or distance code; a dynamic block may have no distance code at all (it then holds literals only, and any
// match is an error); HLIT <= 286, HDIST <= 30; the end-of-block code must have a length; fixed-code symbols 286, 287 and
// distance symbols 30, 31 are invalid when they occur.  The DEFLATE data must end exactly at the end of the member's payload
// (where its trailer starts), as gzip requires.
//
// Safety: every input read is checked against the member's payload, every output write against [out_offset, out_offset + isize);
// corrupt input sets the member's status (PHM_INFLATE_*) and never makes an out-of-bounds access.
#include "phm_common.cuh"

namespace phm {
namespace inflate {

constexpr int WARPS = 8;                 // members per CTA
constexpr int LIT_BITS = 10, DIST_BITS = 8, CL_BITS = 7;
constexpr int MAX_BITS = 15;

struct WarpTables {                      // 4 040 bytes per warp
    uint16_t lit[1 << LIT_BITS];         // primary entries: (symbol << 4) | length, 0 = longer code or no code
    uint16_t dist[1 << DIST_BITS];
    uint16_t cl[1 << CL_BITS];
    uint16_t lit_sorted[288], dist_sorted[32], cl_sorted[20];
    uint16_t lit_count[16], dist_count[16], cl_count[16];
    int32_t run[16], code_base[16];      // table build scratch
    uint8_t lens[320];                   // code lengths of the block's lit/len (0..287) and distance (nlen..) symbols
};

struct Table {                           // one code in shared memory
    uint16_t *prim, *count, *sorted;
    int bits;
};

__constant__ uint16_t LEN_BASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31,
                                      35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t LEN_EXTRA[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t DIST_BASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193,
                                       257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t DIST_EXTRA[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t CL_ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// The input of one member: a bit buffer in registers, every lane holding the same value.
struct Bits {
    const uint8_t *src;
    int64_t len, pos;                    // payload bytes, next byte to load
    uint64_t buf;
    int cnt;                             // valid bits in buf

    __device__ __forceinline__ void refill() {
        if (cnt <= 56) {
            int take = (63 - cnt) >> 3;
            if (take > len - pos) take = (int)(len - pos);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < take) buf |= (uint64_t)__ldg(src + pos + i) << (cnt + 8 * i);
            pos += take;
            cnt += 8 * take;
        }
    }
    // n <= 32 bits; false when the payload ends first
    __device__ __forceinline__ bool take(int n, uint32_t &v) {
        if (cnt < n) refill();
        if (cnt < n) return false;
        v = (uint32_t)(buf & ((1ull << n) - 1ull));
        buf >>= n;
        cnt -= n;
        return true;
    }
};

// Huffman decode of one symbol: >= 0 the symbol, else -PHM_INFLATE_* status
__device__ __forceinline__ int decode(Bits &in, const Table &t) {
    in.refill();
    const uint32_t e = t.prim[in.buf & ((1u << t.bits) - 1u)];
    if (e != 0u) {
        const int n = (int)(e & 15u);
        if (n > in.cnt) return -PHM_INFLATE_TRUNCATED;
        in.buf >>= n;
        in.cnt -= n;
        return (int)(e >> 4);
    }
    int code = 0, first = 0, index = 0;                       // longer than the primary table: one bit at a time (puff.c)
    for (int n = 1; n <= MAX_BITS; ++n) {
        if (n > in.cnt) return -PHM_INFLATE_TRUNCATED;
        code |= (int)((in.buf >> (n - 1)) & 1u);
        const int count = t.count[n];
        if (code - count < first) {
            in.buf >>= n;
            in.cnt -= n;
            return t.sorted[index + (code - first)];
        }
        index += count;
        first = (first + count) << 1;
        code <<= 1;
    }
    return -PHM_INFLATE_BAD_CODE;
}

// Builds the code of lens[0, n) into t (the whole warp; lens are in shared memory).  kind 0 = code-length code, 1 = lit/len or
// distance code.  Returns 0 or PHM_INFLATE_BAD_CODE (over-subscribed; incomplete beyond what zlib accepts; code-length code empty).
__device__ int build(const uint8_t *lens, int n, const Table &t, int kind, WarpTables &w) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    if (lane < 16) t.count[lane] = 0;
    for (int i = lane; i < (1 << t.bits); i += 32) t.prim[i] = 0;
    __syncwarp();
    for (int s0 = 0; s0 < n; s0 += 32) {                        // count[len]: lanes of one length in a chunk add once
        const int s = s0 + lane;
        const uint32_t L = s < n ? lens[s] : 0u;
        const uint32_t m = __match_any_sync(FULL, L);
        if (L != 0u && lane == __ffs(m) - 1) t.count[L] += (uint16_t)__popc(m);
        __syncwarp();
    }
    // canonical codes (RFC 1951 3.2.2), and the checks zlib's inflate_table makes
    int left = 1, max_len = 0, offs = 0, code = 0, my_base = 0, my_off = 0;
    for (int len = 1; len <= MAX_BITS; ++len) {
        const int c = t.count[len];
        left = (left << 1) - c;
        if (left < 0) return PHM_INFLATE_BAD_CODE;              // over-subscribed
        if (c) max_len = len;
        if (len == lane) { my_off = offs; my_base = code - offs; }  // code of the symbol with sorted index i of this length: i + base
        offs += c;
        code = (code + c) << 1;
    }
    if (max_len == 0 && kind == 0) return PHM_INFLATE_BAD_CODE;
    if (left > 0 && max_len != 0 && (kind == 0 || max_len != 1)) return PHM_INFLATE_BAD_CODE;  // incomplete
    __syncwarp();
    if (lane >= 1 && lane <= MAX_BITS) { w.run[lane] = my_off; w.code_base[lane] = my_base; }
    __syncwarp();
    for (int s0 = 0; s0 < n; s0 += 32) {                        // sorted symbols and primary entries, in symbol order per length
        const int s = s0 + lane;
        const uint32_t L = s < n ? lens[s] : 0u;
        const uint32_t m = __match_any_sync(FULL, L);
        const int rank = __popc(m & ((1u << lane) - 1u));
        const int idx = L ? w.run[L] + rank : 0;
        __syncwarp();
        if (L != 0u) {
            if (lane == __ffs(m) - 1) w.run[L] += __popc(m);
            t.sorted[idx] = (uint16_t)s;
            if ((int)L <= t.bits) {
                const uint32_t c = (uint32_t)(idx + w.code_base[L]);
                const uint32_t rev = __brev(c) >> (32 - L);     // codes are sent most significant bit first
                for (uint32_t j = rev; j < (1u << t.bits); j += 1u << L) t.prim[j] = (uint16_t)((s << 4) | (int)L);
            }
        }
        __syncwarp();
    }
    return 0;
}

// ---- CRC32 (gzip's, reflected 0xEDB88320) ----
constexpr uint32_t POLY = 0xEDB88320u;
__device__ __forceinline__ uint32_t multmodp(uint32_t a, uint32_t b) {   // a * b modulo the CRC polynomial (zlib crc32.c)
    uint32_t m = 1u << 31, p = 0u;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1u)) == 0u) break;
        }
        m >>= 1;
        b = (b & 1u) ? (b >> 1) ^ POLY : b >> 1;
    }
    return p;
}
// x^(8 n) modulo the polynomial: the factor that moves a CRC past n more bytes (s_x2n[k] = x^(2^k))
__device__ __forceinline__ uint32_t x8nmodp(uint32_t n, const uint32_t *s_x2n) {
    uint32_t p = 1u << 31;
    for (int k = 3; n; n >>= 1, ++k)
        if (n & 1u) p = multmodp(s_x2n[k & 31], p);
    return p;
}

__global__ void __launch_bounds__(WARPS * 32) inflate_kernel(const uint8_t *__restrict__ in, const phm_bgzf_member *__restrict__ members,
                                                             int64_t n_members, uint8_t *__restrict__ out, int32_t *__restrict__ status,
                                                             unsigned long long *__restrict__ first_bad) {
    __shared__ WarpTables s_tab[WARPS];
    __shared__ uint32_t s_crc[256], s_x2n[32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t c = (uint32_t)i;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ POLY : c >> 1;
        s_crc[i] = c;
    }
    if (threadIdx.x == 0) {
        uint32_t p = 1u << 30;                                   // x^1
        s_x2n[0] = p;
        for (int k = 1; k < 32; ++k) s_x2n[k] = p = multmodp(p, p);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WarpTables &w = s_tab[wid];
    const Table lit = {w.lit, w.lit_count, w.lit_sorted, LIT_BITS};
    const Table dist = {w.dist, w.dist_count, w.dist_sorted, DIST_BITS};
    const Table cl = {w.cl, w.cl_count, w.cl_sorted, CL_BITS};
    for (int64_t mi = (int64_t)blockIdx.x * WARPS + wid; mi < n_members; mi += (int64_t)gridDim.x * WARPS) {
        const phm_bgzf_member mem = members[mi];
        uint8_t *dst = out + mem.out_offset;
        const int64_t isize = mem.isize;
        Bits bits;
        bits.src = in + mem.in_offset; bits.len = mem.in_bytes; bits.pos = 0; bits.buf = 0ull; bits.cnt = 0;
        int64_t o = 0;                                           // bytes written
        int st = 0;
        uint32_t bfinal = 0u;
        do {
            uint32_t hdr;
            if (!bits.take(3, hdr)) { st = PHM_INFLATE_TRUNCATED; break; }
            bfinal = hdr & 1u;
            const uint32_t btype = hdr >> 1;
            if (btype == 0u) {                                   // stored: LEN, NLEN from the next byte boundary
                const int drop = bits.cnt & 7;
                bits.buf >>= drop; bits.cnt -= drop;
                uint32_t len, nlen;
                if (!bits.take(16, len) || !bits.take(16, nlen)) { st = PHM_INFLATE_TRUNCATED; break; }
                if ((len ^ 0xFFFFu) != nlen) { st = PHM_INFLATE_STORED_LEN; break; }
                const int64_t at = bits.pos - (bits.cnt >> 3);   // the bytes still in the bit buffer are the block's first ones
                bits.pos = at; bits.buf = 0ull; bits.cnt = 0;
                if (at + len > bits.len) { st = PHM_INFLATE_TRUNCATED; break; }
                if (o + len > isize) { st = PHM_INFLATE_OVERFLOW; break; }
                __syncwarp();
                for (uint32_t i = lane; i < len; i += 32) dst[o + i] = __ldg(bits.src + at + i);
                bits.pos = at + len;
                o += len;
                __syncwarp();
                continue;
            }
            if (btype == 3u) { st = PHM_INFLATE_BTYPE; break; }
            if (btype == 1u) {                                   // fixed codes (RFC 1951 3.2.6); 286, 287 and 30, 31 are invalid
                __syncwarp();
                for (int i = lane; i < 320; i += 32)
                    w.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
                build(w.lens, 288, lit, 1, w);
                build(w.lens + 288, 32, dist, 1, w);
            } else {                                             // dynamic codes (RFC 1951 3.2.7)
                uint32_t h;
                if (!bits.take(14, h)) { st = PHM_INFLATE_TRUNCATED; break; }
                const int nlen = 257 + (int)(h & 31u), ndist = 1 + (int)((h >> 5) & 31u), ncode = 4 + (int)(h >> 10);
                if (nlen > 286 || ndist > 30) { st = PHM_INFLATE_BAD_CODE; break; }
                __syncwarp();
                if (lane < 19) w.lens[lane] = 0;
                __syncwarp();
                for (int i = 0; i < ncode; ++i) {
                    uint32_t v;
                    if (!bits.take(3, v)) { st = PHM_INFLATE_TRUNCATED; break; }
                    if (lane == 0) w.lens[CL_ORDER[i]] = (uint8_t)v;
                }
                if (st) break;
                if (build(w.lens, 19, cl, 0, w)) { st = PHM_INFLATE_BAD_CODE; break; }
                // the code lengths of lit/len and distance symbols, as one sequence (repeats may cross from one to the other)
                int idx = 0, prev = -1;
                while (idx < nlen + ndist) {
                    const int sym = decode(bits, cl);
                    if (sym < 0) { st = -sym; break; }
                    if (sym < 16) {
                        if (lane == 0) w.lens[idx] = (uint8_t)sym;
                        prev = sym;
                        ++idx;
                        continue;
                    }
                    uint32_t rep, v;
                    int val = 0;
                    if (sym == 16) {
                        if (prev < 0) { st = PHM_INFLATE_BAD_CODE; break; }
                        val = prev;
                        if (!bits.take(2, v)) { st = PHM_INFLATE_TRUNCATED; break; }
                        rep = 3u + v;
                    } else if (sym == 17) {
                        if (!bits.take(3, v)) { st = PHM_INFLATE_TRUNCATED; break; }
                        rep = 3u + v;
                    } else {
                        if (!bits.take(7, v)) { st = PHM_INFLATE_TRUNCATED; break; }
                        rep = 11u + v;
                    }
                    if (idx + (int)rep > nlen + ndist) { st = PHM_INFLATE_BAD_CODE; break; }
                    for (uint32_t i = lane; i < rep; i += 32) w.lens[idx + i] = (uint8_t)val;
                    prev = val;
                    idx += (int)rep;
                }
                if (st) break;
                __syncwarp();
                if (w.lens[256] == 0) { st = PHM_INFLATE_BAD_CODE; break; }   // no end-of-block code
                if (build(w.lens, nlen, lit, 1, w) || build(w.lens + nlen, ndist, dist, 1, w)) { st = PHM_INFLATE_BAD_CODE; break; }
            }
            for (;;) {                                           // the block's symbols
                const int sym = decode(bits, lit);
                if (sym < 0) { st = -sym; break; }
                if (sym < 256) {
                    if (o >= isize) { st = PHM_INFLATE_OVERFLOW; break; }
                    if (lane == 0) dst[o] = (uint8_t)sym;
                    ++o;
                    continue;
                }
                if (sym == 256) break;
                if (sym > 285) { st = PHM_INFLATE_BAD_CODE; break; }
                uint32_t v;
                if (!bits.take(LEN_EXTRA[sym - 257], v)) { st = PHM_INFLATE_TRUNCATED; break; }
                const int len = LEN_BASE[sym - 257] + (int)v;
                const int ds = decode(bits, dist);
                if (ds < 0) { st = -ds; break; }
                if (ds > 29) { st = PHM_INFLATE_BAD_CODE; break; }
                if (!bits.take(DIST_EXTRA[ds], v)) { st = PHM_INFLATE_TRUNCATED; break; }
                const int d = DIST_BASE[ds] + (int)v;
                if (d > o) { st = PHM_INFLATE_DISTANCE; break; }
                if (o + len > isize) { st = PHM_INFLATE_OVERFLOW; break; }
                __syncwarp();                                    // lane 0's literals are visible to the warp
                uint8_t *p = dst + o;
                if (d >= len) {
                    for (int i = lane; i < len; i += 32) p[i] = p[i - d];
                } else {                                         // overlapping: the d bytes before repeat
                    for (int i = lane; i < len; i += 32) p[i] = p[i % d - d];
                }
                o += len;
                __syncwarp();
            }
        } while (!st && !bfinal);
        if (!st && bits.pos - (bits.cnt >> 3) != bits.len) st = PHM_INFLATE_TRAILING;
        if (!st && o != isize) st = PHM_INFLATE_ISIZE;
        __syncwarp();
        if (!st) {                                               // CRC32: lane j takes a contiguous piece; pieces are combined
            const int64_t piece = (isize + 31) / 32, lo = lane * piece < isize ? lane * piece : isize;
            const int64_t hi = lo + piece < isize ? lo + piece : isize;
            uint32_t c = 0xFFFFFFFFu;
            for (int64_t i = lo; i < hi; ++i) c = s_crc[(c ^ dst[i]) & 255u] ^ (c >> 8);
            c = ~c;                                              // gzip's CRC of the piece
            c = hi > lo ? multmodp(x8nmodp((uint32_t)(isize - hi), s_x2n), c) : 0u;   // moved past the bytes after it
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) c ^= __shfl_xor_sync(FULL, c, off);
            if (c != mem.crc32) st = PHM_INFLATE_CRC;
        }
        if (lane == 0) {
            status[mi] = st;
            if (st) atomicMin(first_bad, ((unsigned long long)mi << 8) | (unsigned long long)st);
        }
    }
}

}  // namespace inflate
}  // namespace phm

using namespace phm;

static const char *inflate_reason(int st) {
    switch (st) {
        case PHM_INFLATE_BTYPE: return "block type 3";
        case PHM_INFLATE_STORED_LEN: return "stored block LEN / NLEN mismatch";
        case PHM_INFLATE_BAD_CODE: return "invalid Huffman code or code lengths";
        case PHM_INFLATE_DISTANCE: return "distance before the member's start";
        case PHM_INFLATE_OVERFLOW: return "output past ISIZE";
        case PHM_INFLATE_TRUNCATED: return "payload ends before the final block";
        case PHM_INFLATE_TRAILING: return "payload continues after the final block";
        case PHM_INFLATE_ISIZE: return "output shorter than ISIZE";
        case PHM_INFLATE_CRC: return "CRC32 mismatch";
        default: return "unknown";
    }
}

extern "C" size_t phm_inflate_workspace_bytes(int64_t n_members) {
    if (n_members < 0) n_members = 0;
    return (((size_t)n_members * sizeof(phm_bgzf_member) + 255) & ~(size_t)255) + 256;
}

extern "C" int phm_inflate(const uint8_t *d_in, int64_t in_bytes, const phm_bgzf_member *h_members, int64_t n_members, uint8_t *d_out,
                           int64_t out_bytes, int32_t *d_status, void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(in_bytes >= 0 && out_bytes >= 0 && n_members >= 0, "negative size");
    PHM_REQUIRE(n_members == 0 || (h_members != nullptr && d_status != nullptr && d_workspace != nullptr), "null pointer");
    PHM_REQUIRE(d_in != nullptr || in_bytes == 0, "d_in is null");
    PHM_REQUIRE(d_out != nullptr || out_bytes == 0, "d_out is null");
    int64_t end = 0;
    for (int64_t i = 0; i < n_members; ++i) {
        const phm_bgzf_member &m = h_members[i];
        if (m.in_bytes > PHM_BGZF_MAX_BYTES || m.isize > PHM_BGZF_MAX_BYTES) {
            set_error("invalid argument: member %lld: payload %u / isize %u bytes is beyond the BGZF limit of %d", (long long)i, m.in_bytes,
                      m.isize, PHM_BGZF_MAX_BYTES);
            return PHM_E_ARG;
        }
        if (m.in_offset < 0 || m.in_offset > in_bytes - (int64_t)m.in_bytes) {
            set_error("invalid argument: member %lld: payload [%lld, +%u) is outside the %lld input bytes", (long long)i,
                      (long long)m.in_offset, m.in_bytes, (long long)in_bytes);
            return PHM_E_ARG;
        }
        if (m.out_offset < end || m.out_offset > out_bytes - (int64_t)m.isize) {
            set_error("invalid argument: member %lld: output [%lld, +%u) overlaps the previous member's or is outside the %lld "
                      "output bytes (outputs must be in ascending order)", (long long)i, (long long)m.out_offset, m.isize,
                      (long long)out_bytes);
            return PHM_E_ARG;
        }
        end = m.out_offset + m.isize;
    }
    const size_t need = phm_inflate_workspace_bytes(n_members);
    if (n_members > 0 && workspace_bytes < need) { set_error("workspace too small: %zu < %zu", workspace_bytes, need); return PHM_E_WORKSPACE; }
    if (n_members == 0) return PHM_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned char *base = static_cast<unsigned char *>(d_workspace);
    phm_bgzf_member *d_members = reinterpret_cast<phm_bgzf_member *>(base);
    unsigned long long *d_first = reinterpret_cast<unsigned long long *>(base + need - 256);
    PHM_CUDA_CHECK(cudaMemcpyAsync(d_members, h_members, (size_t)n_members * sizeof(phm_bgzf_member), cudaMemcpyHostToDevice, st));
    PHM_CUDA_CHECK(cudaMemsetAsync(d_first, 0xFF, sizeof(unsigned long long), st));
    int64_t grid = (n_members + inflate::WARPS - 1) / inflate::WARPS;
    const int64_t cap = (int64_t)sm_count() * 32;
    if (grid > cap) grid = cap;
    inflate::inflate_kernel<<<(unsigned)grid, inflate::WARPS * 32, 0, st>>>(d_in, d_members, n_members, d_out, d_status, d_first);
    PHM_LAUNCH_CHECK();
    unsigned long long first = 0;
    PHM_CUDA_CHECK(cudaMemcpyAsync(&first, d_first, sizeof(first), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (first != ~0ull) {
        const int code = (int)(first & 255ull);
        set_error("corrupt DEFLATE data: member %lld: %s (status %d)", (long long)(first >> 8), inflate_reason(code), code);
        return PHM_E_DATA;
    }
    return PHM_OK;
}
