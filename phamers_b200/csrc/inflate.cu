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
// The decode tables and what is accepted (zlib's rules) are described in inflate_common.cuh.  The DEFLATE data must end exactly
// at the end of the member's payload (where its trailer starts), as gzip requires.  gunzip.cu's read_dynamic and decode_span
// repeat this kernel's header reader and block loop: a change to what is accepted must be made in both.
//
// Safety: every input read is checked against the member's payload, every output write against [out_offset, out_offset + isize);
// corrupt input sets the member's status (PHM_INFLATE_*) and never makes an out-of-bounds access.
#include "inflate_common.cuh"

namespace phm {
namespace inflate {

constexpr int WARPS = 8;                 // members per CTA

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
