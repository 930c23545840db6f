// The RFC 1951 pieces shared by the DEFLATE decoders (inflate.cu: BGZF members; gunzip.cu: one gzip member decoded in chunks):
// the input bit buffer, Huffman decode and table build in a warp's shared memory, the length / distance tables, and gzip's CRC32
// with zlib's combination of piece CRCs.
//
// Decode tables (RFC 1951 canonical codes): a primary table indexed by the next LIT_BITS / DIST_BITS / CL_BITS input bits gives
// (symbol, length) for every code no longer than that; a longer code (rare: lit/len codes of 11..15 bits, distance codes of
// 9..15) is decoded bit by bit from the per-length counts and the symbols sorted by code (the method of zlib's puff.c).
// The code-length code has at most 7 bits and is always decoded from its primary table.
//
// What is accepted is what zlib accepts: an over-subscribed code is an error; an incomplete code only when it is a single code of
// one bit in a lit/len or distance code; a dynamic block may have no distance code at all (it then holds literals only, and any
// match is an error); HLIT <= 286, HDIST <= 30; the end-of-block code must have a length; fixed-code symbols 286, 287 and
// distance symbols 30, 31 are invalid when they occur.
#pragma once
#include "phm_common.cuh"

namespace phm {
namespace inflate {

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
static __device__ int build(const uint8_t *lens, int n, const Table &t, int kind, WarpTables &w) {
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

}  // namespace inflate
}  // namespace phm
