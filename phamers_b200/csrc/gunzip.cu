// Single-member gzip decompression on the device: the DEFLATE stream of an ordinary .gz file (gzip, pigz) is decoded in parallel
// although nothing tells where its blocks start or what they output (the approach of pugz / rapidgzip).  The payload is cut into
// chunks of `gunzip_chunk_bytes` compressed bytes, and
//
//   finder   for every chunk but the first, one warp finds the first bit offset at or after the chunk's start where a dynamic
//            block header validates completely (BTYPE 10; HLIT, HDIST <= 29; a complete code-length code; the code lengths
//            decode without overrun and a repeat 16 never comes first; the end-of-block code has a length; both codes build).
//            Each lane first screens 8 offsets on their first 74 bits (the block type, HLIT, HDIST and the code-length code's Kraft
//            sum); the warp then validates the survivors in offset order.  Stored and fixed blocks are not searched for: a chunk
//            without a candidate is covered by its predecessor's decoder.
//   pass A   one warp per candidate decodes from it, counting output without writing it, and stops at the first block end at or
//            after the next candidate (or at the final block).  A link is verified when its predecessor is verified and ended
//            exactly at its start; chunk 0 starts at bit 0.  A candidate inside a verified link's range was false; the link
//            after a mismatch is decoded again from the verified end (a repair round; later mismatches are repaired in the same
//            round, speculatively).  An error in a verified link means the stream is corrupt; in an unverified one, only that its
//            candidate was false.  After MAX_ROUNDS rounds, one warp decodes the rest of the stream from the last verified end.
//   pass B   the prefix sum of the verified links' lengths places each link's output.  Each link is decoded again into uint16
//            symbols: a byte as itself, a byte that a match copies from before the link's first byte as 0x8000 | its position in
//            the 32 KiB window before the link (a copy of such a marker copies the marker, so markers never chain).
//   pass C   literal symbols go to the output; then one CTA walks the links in file order and resolves the markers in each link's
//            last 32 KiB (the only bytes a later link's window can see), which makes every window complete; a link whose markers
//            all lie before its last 32 KiB costs that walk nothing.  Then all other markers resolve in parallel.  Pass C runs
//            only when every link decoded cleanly in pass B.  The CRC32 is computed in pieces and combined (zlib's
//            crc32_combine); ISIZE and the end of the stream (the trailer must follow it exactly) are checked by the index call.
//
// The chain walk runs on the host between rounds (a few bytes per chunk cross PCIe).  The output is exactly what zlib gives
// whenever the call succeeds: every verified link starts on a true block boundary, and any disagreement with zlib's rules, the
// trailer's CRC32 or ISIZE, or bytes after the final block is PHM_E_DATA.  Every input read is bounds-checked against the payload
// and every write against its link's output range, whatever the bits say.
#include <algorithm>
#include <vector>

#include "inflate_common.cuh"

namespace phm {
namespace gunzip {
using namespace inflate;

constexpr int WARPS = 8;                 // chunks (links) per CTA
constexpr int MAX_ROUNDS = 16;           // repair rounds before the rest of the stream is decoded serially
constexpr int64_t NO_STOP = INT64_MAX;   // decode to the final block
constexpr int RESOLVE_THREADS = 1024;

struct Link {                            // one verified piece of the stream (index workspace)
    int64_t start, end;                  // bit range of the payload
    int64_t len, off;                    // output bytes, offset in the output
    int64_t last_marker;                 // written by pass B: last output index (relative) holding a window marker, or -1
};

struct Header {                          // first bytes of the index workspace
    int64_t n_links, total, payload_bytes, n_chunks;
};

struct Span {
    int64_t end, len, last_marker;
    int status, final;
};

int chunk_bytes = 128 << 10;             // option "gunzip_chunk_bytes" (1 KiB .. 1 GiB)

// The dynamic block header after BTYPE (RFC 1951 3.2.7): tables built into lit / dist.  0 or a PHM_INFLATE_* status.  This and
// the block loop of decode_span follow inflate_kernel (inflate.cu) line for line, which keeps its own copy so that its code stays
// as measured; a change to what is accepted must be made in both.
__device__ __forceinline__ int read_dynamic(Bits &bits, WarpTables &w, const Table &lit, const Table &dist, const Table &cl) {
    const int lane = threadIdx.x & 31;
    uint32_t h;
    if (!bits.take(14, h)) return PHM_INFLATE_TRUNCATED;
    const int nlen = 257 + (int)(h & 31u), ndist = 1 + (int)((h >> 5) & 31u), ncode = 4 + (int)(h >> 10);
    if (nlen > 286 || ndist > 30) return PHM_INFLATE_BAD_CODE;
    __syncwarp();
    if (lane < 19) w.lens[lane] = 0;
    __syncwarp();
    for (int i = 0; i < ncode; ++i) {
        uint32_t v;
        if (!bits.take(3, v)) return PHM_INFLATE_TRUNCATED;
        if (lane == 0) w.lens[CL_ORDER[i]] = (uint8_t)v;
    }
    if (build(w.lens, 19, cl, 0, w)) return PHM_INFLATE_BAD_CODE;
    int idx = 0, prev = -1;
    while (idx < nlen + ndist) {
        const int sym = decode(bits, cl);
        if (sym < 0) return -sym;
        if (sym < 16) {
            if (lane == 0) w.lens[idx] = (uint8_t)sym;
            prev = sym;
            ++idx;
            continue;
        }
        uint32_t rep, v;
        int val = 0;
        if (sym == 16) {
            if (prev < 0) return PHM_INFLATE_BAD_CODE;
            val = prev;
            if (!bits.take(2, v)) return PHM_INFLATE_TRUNCATED;
            rep = 3u + v;
        } else if (sym == 17) {
            if (!bits.take(3, v)) return PHM_INFLATE_TRUNCATED;
            rep = 3u + v;
        } else {
            if (!bits.take(7, v)) return PHM_INFLATE_TRUNCATED;
            rep = 11u + v;
        }
        if (idx + (int)rep > nlen + ndist) return PHM_INFLATE_BAD_CODE;
        for (uint32_t i = lane; i < rep; i += 32) w.lens[idx + i] = (uint8_t)val;
        prev = val;
        idx += (int)rep;
    }
    __syncwarp();
    if (w.lens[256] == 0) return PHM_INFLATE_BAD_CODE;          // no end-of-block code
    if (build(w.lens, nlen, lit, 1, w) || build(w.lens + nlen, ndist, dist, 1, w)) return PHM_INFLATE_BAD_CODE;
    return 0;
}

// The bit buffer positioned at bit `start` of the payload; false when that is past its end.
__device__ __forceinline__ bool seek(Bits &bits, const uint8_t *src, int64_t n_bytes, int64_t start) {
    bits.src = src; bits.len = n_bytes; bits.pos = start >> 3; bits.buf = 0ull; bits.cnt = 0;
    uint32_t v;
    if (start < 0 || bits.pos > n_bytes) return false;
    return (start & 7) == 0 || bits.take((int)(start & 7), v);
}

// The whole warp decodes blocks from bit `start` until a block ends at or after bit `stop`, or the final block ends.  SYMBOLS:
// the output goes to sym[0, cap) as symbols (see the top of the file), else it is only counted.  known_off >= 0: the output
// offset of the first byte, so that a match reaching before the stream's start is PHM_INFLATE_DISTANCE.
template <bool SYMBOLS>
__device__ __forceinline__ Span decode_span(const uint8_t *__restrict__ src, int64_t n_bytes, int64_t start, int64_t stop, int64_t known_off,
                            uint16_t *__restrict__ sym, int64_t cap, WarpTables &w, const Table &lit, const Table &dist,
                            const Table &cl) {
    const int lane = threadIdx.x & 31;
    Bits bits;
    int64_t o = 0, mark = -1, end = start;
    int st = seek(bits, src, n_bytes, start) ? 0 : PHM_INFLATE_TRUNCATED;
    uint32_t bfinal = 0u;
    while (!st) {
        uint32_t hdr;
        if (!bits.take(3, hdr)) { st = PHM_INFLATE_TRUNCATED; break; }
        bfinal = hdr & 1u;
        const uint32_t btype = hdr >> 1;
        if (btype == 0u) {                                       // stored: LEN, NLEN from the next byte boundary
            const int drop = bits.cnt & 7;
            bits.buf >>= drop; bits.cnt -= drop;
            uint32_t len, nlen;
            if (!bits.take(16, len) || !bits.take(16, nlen)) { st = PHM_INFLATE_TRUNCATED; break; }
            if ((len ^ 0xFFFFu) != nlen) { st = PHM_INFLATE_STORED_LEN; break; }
            const int64_t at = bits.pos - (bits.cnt >> 3);
            bits.pos = at; bits.buf = 0ull; bits.cnt = 0;
            if (at + len > bits.len) { st = PHM_INFLATE_TRUNCATED; break; }
            if (SYMBOLS) {
                if (o + len > cap) { st = PHM_INFLATE_OVERFLOW; break; }
                __syncwarp();
                for (uint32_t i = lane; i < len; i += 32) sym[o + i] = __ldg(src + at + i);
                __syncwarp();
            }
            bits.pos = at + len;
            o += len;
        } else if (btype == 3u) {
            st = PHM_INFLATE_BTYPE;
            break;
        } else {
            if (btype == 1u) {                                   // fixed codes (RFC 1951 3.2.6)
                __syncwarp();
                for (int i = lane; i < 320; i += 32)
                    w.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
                build(w.lens, 288, lit, 1, w);
                build(w.lens + 288, 32, dist, 1, w);
            } else if ((st = read_dynamic(bits, w, lit, dist, cl)) != 0) {
                break;
            }
            for (;;) {                                           // the block's symbols
                const int s = decode(bits, lit);
                if (s < 0) { st = -s; break; }
                if (s < 256) {
                    if (SYMBOLS) {
                        if (o >= cap) { st = PHM_INFLATE_OVERFLOW; break; }
                        if (lane == 0) sym[o] = (uint16_t)s;
                    }
                    ++o;
                    continue;
                }
                if (s == 256) break;
                if (s > 285) { st = PHM_INFLATE_BAD_CODE; break; }
                uint32_t v;
                if (!bits.take(LEN_EXTRA[s - 257], v)) { st = PHM_INFLATE_TRUNCATED; break; }
                const int len = LEN_BASE[s - 257] + (int)v;
                const int ds = decode(bits, dist);
                if (ds < 0) { st = -ds; break; }
                if (ds > 29) { st = PHM_INFLATE_BAD_CODE; break; }
                if (!bits.take(DIST_EXTRA[ds], v)) { st = PHM_INFLATE_TRUNCATED; break; }
                const int d = DIST_BASE[ds] + (int)v;
                if (known_off >= 0 && d > known_off + o) { st = PHM_INFLATE_DISTANCE; break; }
                if (SYMBOLS) {
                    if (o + len > cap) { st = PHM_INFLATE_OVERFLOW; break; }
                    __syncwarp();                                // lane 0's literals are visible to the warp
                    for (int i = lane; i < len; i += 32) {
                        const int64_t rel = o - d + (d >= len ? i : i % d);     // the source, always before o
                        const uint16_t x = rel >= 0 ? sym[rel] : (uint16_t)(0x8000 | (32768 + rel));
                        sym[o + i] = x;
                        if (x & 0x8000u) mark = o + i;
                    }
                    __syncwarp();
                }
                o += len;
            }
            if (st) break;
        }
        end = bits.pos * 8 - bits.cnt;                           // this block's end
        if (bfinal || end >= stop) break;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const int64_t m = __shfl_xor_sync(FULL, mark, off);
        mark = m > mark ? m : mark;
    }
    Span r;
    r.end = end; r.len = o; r.last_marker = mark; r.status = st; r.final = !st && bfinal;
    return r;
}

__device__ __forceinline__ void warp_tables(WarpTables &w, Table &lit, Table &dist, Table &cl) {
    lit = {w.lit, w.lit_count, w.lit_sorted, LIT_BITS};
    dist = {w.dist, w.dist_count, w.dist_sorted, DIST_BITS};
    cl = {w.cl, w.cl_count, w.cl_sorted, CL_BITS};
}

// Finder: start[c] = the first bit of chunk c (c >= 1) where a dynamic block header validates, or -1.
__global__ void __launch_bounds__(WARPS * 32, 4) gunzip_find_kernel(const uint8_t *__restrict__ src, int64_t n_bytes, int64_t n_chunks,
                                                                 int64_t chunk, int64_t *__restrict__ start) {
    __shared__ WarpTables s_tab[WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WarpTables &w = s_tab[wid];
    Table lit, dist, cl;
    warp_tables(w, lit, dist, cl);
    for (int64_t c = 1 + (int64_t)blockIdx.x * WARPS + wid; c < n_chunks; c += (int64_t)gridDim.x * WARPS) {
        const int64_t lo = c * chunk, hi = lo + chunk < n_bytes ? lo + chunk : n_bytes;
        int64_t found = -1;
        for (int64_t b0 = lo; b0 < hi && found < 0; b0 += 32) {
            const int64_t b = b0 + lane;                         // this lane screens the 8 offsets of byte b
            uint32_t mask = 0u;
            if (b < hi) {
                uint64_t x0 = 0ull, x1 = 0ull;                   // bytes b .. b + 11, zero past the payload
#pragma unroll
                for (int i = 0; i < 8; ++i) if (b + i < n_bytes) x0 |= (uint64_t)__ldg(src + b + i) << (8 * i);
#pragma unroll
                for (int i = 0; i < 4; ++i) if (b + 8 + i < n_bytes) x1 |= (uint64_t)__ldg(src + b + 8 + i) << (8 * i);
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const uint64_t w0 = s ? (x0 >> s) | (x1 << (64 - s)) : x0;
                    if (((w0 >> 1) & 3u) != 2u || ((w0 >> 3) & 31u) > 29u || ((w0 >> 8) & 31u) > 29u) continue;
                    const int ncode = 4 + (int)((w0 >> 13) & 15u);
                    const uint64_t w1 = (x0 >> (s + 17)) | (x1 << (47 - s));     // the code-length code's lengths
                    uint32_t kraft = 0u;
#pragma unroll
                    for (int k = 0; k < 19; ++k) {
                        const uint32_t l = (uint32_t)(w1 >> (3 * k)) & 7u;
                        if (k < ncode && l) kraft += 128u >> l;
                    }
                    if (kraft == 128u) mask |= 1u << s;          // complete (zlib rejects any other code-length code)
                }
            }
            uint32_t any = __ballot_sync(FULL, mask != 0u);
            while (any && found < 0) {
                const int l = __ffs(any) - 1;
                any &= any - 1u;
                uint32_t m = __shfl_sync(FULL, mask, l);
                while (m) {
                    const int s = __ffs(m) - 1;
                    m &= m - 1u;
                    const int64_t p = (b0 + l) * 8 + s;
                    Bits bits;
                    uint32_t hdr;
                    if (seek(bits, src, n_bytes, p) && bits.take(3, hdr) && (hdr >> 1) == 2u && read_dynamic(bits, w, lit, dist, cl) == 0) {
                        found = p;
                        break;
                    }
                }
            }
        }
        if (lane == 0) start[c] = found;
    }
}

// Pass A (and the repair rounds): the slots of `list` decode from start[j] to the first block end >= stop[j], counting output.
__global__ void __launch_bounds__(WARPS * 32, 4) gunzip_size_kernel(const uint8_t *__restrict__ src, int64_t n_bytes,
                                                                 const int32_t *__restrict__ list, int64_t n_list,
                                                                 const int64_t *__restrict__ start, const int64_t *__restrict__ stop,
                                                                 int64_t *__restrict__ end, int64_t *__restrict__ len,
                                                                 int32_t *__restrict__ status, int32_t *__restrict__ final) {
    __shared__ WarpTables s_tab[WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WarpTables &w = s_tab[wid];
    Table lit, dist, cl;
    warp_tables(w, lit, dist, cl);
    for (int64_t t = (int64_t)blockIdx.x * WARPS + wid; t < n_list; t += (int64_t)gridDim.x * WARPS) {
        const int j = list[t];
        const int64_t s0 = start[j];
        const Span r = decode_span<false>(src, n_bytes, s0, stop[j], s0 == 0 ? 0 : -1, nullptr, 0, w, lit, dist, cl);
        if (lane == 0) { end[j] = r.end; len[j] = r.len; status[j] = r.status; final[j] = r.final; }
    }
}

// Pass B: every link decoded again into its symbols at sym[off, off + len).
__global__ void __launch_bounds__(WARPS * 32, 4) gunzip_symbol_kernel(const uint8_t *__restrict__ src, int64_t n_bytes,
                                                                   Link *__restrict__ links, int64_t n_links, uint16_t *__restrict__ sym,
                                                                   unsigned long long *__restrict__ first_bad) {
    __shared__ WarpTables s_tab[WARPS];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WarpTables &w = s_tab[wid];
    Table lit, dist, cl;
    warp_tables(w, lit, dist, cl);
    for (int64_t j = (int64_t)blockIdx.x * WARPS + wid; j < n_links; j += (int64_t)gridDim.x * WARPS) {
        const Link L = links[j];
        const Span r = decode_span<true>(src, n_bytes, L.start, L.end, L.off, sym + L.off, L.len, w, lit, dist, cl);
        int st = r.status;
        if (!st && (r.end != L.end || r.len != L.len)) st = PHM_INFLATE_BAD_CODE;   // not the decode pass A verified
        if (lane == 0) {
            links[j].last_marker = r.last_marker;
            if (st) atomicMin(first_bad, ((unsigned long long)j << 8) | (unsigned long long)st);
        }
    }
}

// Pass C, 1: literal symbols to the output (marker positions get a placeholder, overwritten below).
__global__ void gunzip_literal_kernel(const uint16_t *__restrict__ sym, int64_t total, uint8_t *__restrict__ out) {
    const int64_t groups = total / 8;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
        const uint4 v = reinterpret_cast<const uint4 *>(sym)[g];
        uint2 b;
        b.x = (v.x & 0xFFu) | ((v.x >> 8) & 0xFF00u) | ((v.y & 0xFFu) << 16) | ((v.y & 0xFF0000u) << 8);
        b.y = (v.z & 0xFFu) | ((v.z >> 8) & 0xFF00u) | ((v.w & 0xFFu) << 16) | ((v.w & 0xFF0000u) << 8);
        reinterpret_cast<uint2 *>(out)[g] = b;
    }
    if (blockIdx.x == 0 && threadIdx.x < total - groups * 8) out[groups * 8 + threadIdx.x] = (uint8_t)sym[groups * 8 + threadIdx.x];
}

__device__ __forceinline__ int64_t tail_start(const Link &L) {   // the link's last 32 KiB: what later windows can see
    const int64_t next = L.off + L.len;
    return next - 32768 > L.off ? next - 32768 : L.off;
}

// The markers among sym[lo, hi) of link L, from the window before it; 8 symbols per thread and step (sym is padded to 8).
__device__ __forceinline__ void resolve_range(const uint16_t *__restrict__ sym, uint8_t *__restrict__ out, int64_t link_off, int64_t lo,
                                              int64_t hi) {
    for (int64_t g = lo / 8 + threadIdx.x; g * 8 < hi; g += blockDim.x) {
        const uint4 v = reinterpret_cast<const uint4 *>(sym)[g];
        const uint32_t words[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint32_t x = (words[q >> 1] >> (16 * (q & 1))) & 0xFFFFu;
            const int64_t i = g * 8 + q;
            const int64_t from = link_off - 32768 + (x & 0x7FFFu);          // before the link; >= 0 after a clean pass B
            if ((x & 0x8000u) && i >= lo && i < hi && from >= 0) out[i] = out[from];
        }
    }
}

// Pass C, 2: one CTA, the links in file order: the markers in each link's last 32 KiB, from the window before it (literals and
// the markers of earlier tails, already resolved).  The link table is read in batches of RESOLVE_THREADS.
__global__ void __launch_bounds__(RESOLVE_THREADS) gunzip_tail_kernel(const Link *__restrict__ links, int64_t n_links,
                                                                      const uint16_t *__restrict__ sym, uint8_t *__restrict__ out) {
    __shared__ int64_t s_off[RESOLVE_THREADS], s_lo[RESOLVE_THREADS], s_hi[RESOLVE_THREADS];
    for (int64_t j0 = 1; j0 < n_links; j0 += RESOLVE_THREADS) {
        const int nb = n_links - j0 < RESOLVE_THREADS ? (int)(n_links - j0) : RESOLVE_THREADS;
        __syncthreads();
        if ((int)threadIdx.x < nb) {
            const Link L = links[j0 + threadIdx.x];
            s_off[threadIdx.x] = L.off;
            s_lo[threadIdx.x] = tail_start(L);
            s_hi[threadIdx.x] = L.off + L.last_marker + 1;
        }
        __syncthreads();
        for (int b = 0; b < nb; ++b) {
            if (s_hi[b] <= s_lo[b]) continue;                   // no marker in the tail: the next window needs nothing from here
            resolve_range(sym, out, s_off[b], s_lo[b], s_hi[b]);
            __syncthreads();
        }
    }
}

// Pass C, 3: every other marker (before its link's tail), 8 symbols per thread and step over the whole output; every window is
// resolved now.  A group holding a marker finds its link by binary search over the link offsets.
__global__ void gunzip_marker_kernel(const Link *__restrict__ links, int64_t n_links, const uint16_t *__restrict__ sym, int64_t total,
                                     uint8_t *__restrict__ out) {
    const int64_t groups = (total + 7) / 8;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
        const uint4 v = reinterpret_cast<const uint4 *>(sym)[g];
        if (((v.x | v.y | v.z | v.w) & 0x80008000u) == 0u) continue;
        const uint32_t words[4] = {v.x, v.y, v.z, v.w};
        int64_t j = -1, next = -1;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint32_t x = (words[q >> 1] >> (16 * (q & 1))) & 0xFFFFu;
            const int64_t i = g * 8 + q;
            if (!(x & 0x8000u) || i >= total) continue;
            if (j < 0 || i >= next) {                            // the link holding i: the last with off <= i
                int64_t lo = 0, hi = n_links - 1;
                while (lo < hi) {
                    const int64_t mid = (lo + hi + 1) / 2;
                    if (links[mid].off <= i) lo = mid; else hi = mid - 1;
                }
                j = lo;
                next = links[j].off + links[j].len;
            }
            const Link L = links[j];
            const int64_t from = L.off - 32768 + (x & 0x7FFFu);
            if (i < tail_start(L) && from >= 0) out[i] = out[from];
        }
    }
}

__device__ __forceinline__ uint32_t x8nmodp64(uint64_t n, const uint32_t *s_x2n) {   // x^(8 n) for a 64-bit n (zlib's x2nmodp)
    uint32_t p = 1u << 31;
    for (int k = 3; n; n >>= 1, ++k)
        if (n & 1u) p = multmodp(s_x2n[k & 31], p);
    return p;
}

// CRC32 of out[0, total): each thread a piece of `piece` bytes (a multiple of 16), moved past the bytes after it and XORed into acc.
__global__ void gunzip_crc_kernel(const uint8_t *__restrict__ out, int64_t total, int64_t piece, uint32_t *__restrict__ acc) {
    __shared__ uint32_t s_crc[256], s_x2n[32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t c = (uint32_t)i;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ POLY : c >> 1;
        s_crc[i] = c;
    }
    if (threadIdx.x == 0) {
        uint32_t p = 1u << 30;
        s_x2n[0] = p;
        for (int k = 1; k < 32; ++k) s_x2n[k] = p = multmodp(p, p);
    }
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t lo = t * piece < total ? t * piece : total, hi = lo + piece < total ? lo + piece : total;
    uint32_t c = 0xFFFFFFFFu;
    int64_t i = lo;
    for (; i + 16 <= hi; i += 16) {
        const uint4 v = *reinterpret_cast<const uint4 *>(out + i);
        const uint32_t words[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int k = 0; k < 4; ++k) c = s_crc[(c ^ (words[q] >> (8 * k))) & 255u] ^ (c >> 8);
    }
    for (; i < hi; ++i) c = s_crc[(c ^ out[i]) & 255u] ^ (c >> 8);
    c = hi > lo ? multmodp(x8nmodp64((uint64_t)(total - hi), s_x2n), ~c) : 0u;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) c ^= __shfl_xor_sync(FULL, c, off);
    if ((threadIdx.x & 31) == 0 && c) atomicXor(acc, c);
}

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

static int64_t n_chunks_of(int64_t payload_bytes, int64_t chunk) {
    return payload_bytes <= chunk ? 1 : (payload_bytes + chunk - 1) / chunk;
}

struct IndexLayout {                     // the index workspace
    Header *hdr;
    int64_t *start, *stop, *end, *len;
    int32_t *status, *final, *list;
    Link *links;
    size_t bytes;
    IndexLayout(void *base, int64_t n) {
        unsigned char *p = static_cast<unsigned char *>(base);
        size_t at = 256;
        auto take = [&](size_t b) { unsigned char *q = p + at; at += align256(b); return q; };
        hdr = reinterpret_cast<Header *>(p);
        start = reinterpret_cast<int64_t *>(take(n * 8)); stop = reinterpret_cast<int64_t *>(take(n * 8));
        end = reinterpret_cast<int64_t *>(take(n * 8)); len = reinterpret_cast<int64_t *>(take(n * 8));
        status = reinterpret_cast<int32_t *>(take(n * 4)); final = reinterpret_cast<int32_t *>(take(n * 4));
        list = reinterpret_cast<int32_t *>(take(n * 4));
        links = reinterpret_cast<Link *>(take(n * sizeof(Link)));
        bytes = at;
    }
};

static int grid_for(int64_t items, int per_cta) {
    int64_t g = (items + per_cta - 1) / per_cta;
    const int64_t cap = (int64_t)sm_count() * 32;
    if (g > cap) g = cap;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace gunzip
}  // namespace phm

using namespace phm;
using namespace phm::gunzip;

static const char *gunzip_reason(int st) {
    switch (st) {
        case PHM_INFLATE_BTYPE: return "block type 3";
        case PHM_INFLATE_STORED_LEN: return "stored block LEN / NLEN mismatch";
        case PHM_INFLATE_BAD_CODE: return "invalid Huffman code or code lengths";
        case PHM_INFLATE_DISTANCE: return "distance before the stream's start";
        case PHM_INFLATE_OVERFLOW: return "output past the link's length";
        case PHM_INFLATE_TRUNCATED: return "payload ends before the final block";
        case PHM_INFLATE_TRAILING: return "payload continues after the final block";
        case PHM_INFLATE_ISIZE: return "output size differs from ISIZE";
        case PHM_INFLATE_CRC: return "CRC32 mismatch";
        default: return "unknown";
    }
}

static int data_error(int st, int64_t at_bit) {
    set_error("corrupt DEFLATE data: %s (status %d) in the piece starting at bit %lld", gunzip_reason(st), st, (long long)at_bit);
    return PHM_E_DATA;
}

extern "C" size_t phm_gunzip_index_workspace_bytes(int64_t payload_bytes) {
    if (payload_bytes < 0) payload_bytes = 0;
    return IndexLayout(nullptr, n_chunks_of(payload_bytes, gunzip::chunk_bytes)).bytes;
}

extern "C" size_t phm_gunzip_extract_workspace_bytes(int64_t out_bytes) {
    if (out_bytes < 0) out_bytes = 0;
    return 256 + align256((size_t)(out_bytes + 8) * sizeof(uint16_t));
}

extern "C" int phm_gunzip_index(const uint8_t *d_payload, int64_t payload_bytes, uint32_t isize, int64_t *h_info, void *d_workspace,
                                size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(payload_bytes >= 0, "negative size");
    PHM_REQUIRE(d_payload != nullptr || payload_bytes == 0, "d_payload is null");
    PHM_REQUIRE(h_info != nullptr && d_workspace != nullptr, "null pointer");
    const int64_t chunk = gunzip::chunk_bytes, n = n_chunks_of(payload_bytes, chunk);
    PHM_REQUIRE(n < INT32_MAX, "too many chunks");
    const IndexLayout ws(d_workspace, n);
    if (workspace_bytes < ws.bytes) { set_error("workspace too small: %zu < %zu", workspace_bytes, ws.bytes); return PHM_E_WORKSPACE; }
    for (int i = 0; i < 7; ++i) h_info[i] = 0;
    h_info[1] = n;
    if (payload_bytes == 0) return data_error(PHM_INFLATE_TRUNCATED, 0);
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    // finder
    std::vector<int64_t> start(n), stop(n), end(n), len(n);
    std::vector<int32_t> status(n), final(n), live(n), list;
    if (n > 1) {
        gunzip_find_kernel<<<grid_for(n - 1, WARPS), WARPS * 32, 0, st>>>(d_payload, payload_bytes, n, chunk, ws.start);
        PHM_LAUNCH_CHECK();
        PHM_CUDA_CHECK(cudaMemcpyAsync(start.data() + 1, ws.start + 1, (n - 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    start[0] = 0;
    const std::vector<int64_t> candidate(start);
    for (int64_t j = 0; j < n; ++j) live[j] = start[j] >= 0;
    for (int64_t j = n - 1, next = NO_STOP; j >= 0; --j) {
        stop[j] = next;
        if (live[j]) { next = start[j]; list.push_back((int32_t)j); }
    }
    std::reverse(list.begin(), list.end());

    // pass A, then repair rounds until the chain is verified from the first bit to the final block
    std::vector<int32_t> chain;
    int64_t rounds = 0;
    for (;;) {
        PHM_CUDA_CHECK(cudaMemcpyAsync(ws.start, start.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        PHM_CUDA_CHECK(cudaMemcpyAsync(ws.stop, stop.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        PHM_CUDA_CHECK(cudaMemcpyAsync(ws.list, list.data(), list.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        gunzip_size_kernel<<<grid_for((int64_t)list.size(), WARPS), WARPS * 32, 0, st>>>(d_payload, payload_bytes, ws.list, (int64_t)list.size(),
                                                                                       ws.start, ws.stop, ws.end, ws.len, ws.status, ws.final);
        PHM_LAUNCH_CHECK();
        PHM_CUDA_CHECK(cudaMemcpyAsync(end.data(), ws.end, n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaMemcpyAsync(len.data(), ws.len, n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaMemcpyAsync(status.data(), ws.status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaMemcpyAsync(final.data(), ws.final, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PHM_CUDA_CHECK(cudaStreamSynchronize(st));

        // the walk: verified links from slot 0; past the first mismatch the walk goes on speculatively, scheduling repairs
        chain.clear();
        list.clear();
        int64_t v = 0;
        bool verified = true, done = false;
        for (;;) {
            if (status[v]) {
                if (verified) return data_error(status[v], start[v]);
                break;                                           // a false candidate's decode: nothing more to infer
            }
            if (verified) chain.push_back((int32_t)v);
            if (final[v]) { done = verified; break; }
            const int64_t e = end[v];
            int64_t k = v + 1;
            while (k < n && (!live[k] || start[k] < e)) live[k++] = 0;   // candidates inside a decoded range were false
            if (k < n && start[k] == e) { v = k; continue; }
            if (v + 1 >= n) {                                   // ended before the final block with nothing after it
                if (verified) return data_error(PHM_INFLATE_TRUNCATED, start[v]);
                break;
            }
            const int64_t r = v + 1;                            // decoded again from e in the next round
            int64_t nx = r + 1;
            while (nx < n && !live[nx]) ++nx;
            start[r] = e; live[r] = 1; stop[r] = nx < n ? start[nx] : NO_STOP;
            list.push_back((int32_t)r);
            verified = false;
            if (nx >= n) break;
            v = nx;
        }
        if (done) break;
        if (rounds >= MAX_ROUNDS) {                              // the rest of the stream by one warp, from the verified end
            const int64_t r = list[0];
            stop[r] = NO_STOP;
            for (int64_t k = r + 1; k < n; ++k) live[k] = 0;
            list.resize(1);
        }
        ++rounds;
    }

    // the verified links, their output offsets and the end-of-stream checks
    std::vector<Link> links(chain.size());
    int64_t total = 0, serial = 0, longest_later = 0;
    const int64_t chunk_bits = chunk * 8;
    for (size_t i = 0; i < chain.size(); ++i) {
        const int64_t j = chain[i];
        links[i] = {start[j], end[j], len[j], total, -1};
        total += len[j];
        if (i > 0 && len[j] > longest_later) longest_later = len[j];
        const int64_t first_whole = (start[j] + chunk_bits - 1) / chunk_bits;
        if ((first_whole + 1) * chunk_bits <= end[j]) serial += len[j];   // spans a chunk that had no link of its own
    }
    int64_t rejected = 0;
    for (int64_t j = 1; j < n; ++j) {
        if (candidate[j] < 0) continue;
        const bool used = std::binary_search(links.begin(), links.end(), Link{candidate[j], 0, 0, 0, 0},
                                             [](const Link &a, const Link &b) { return a.start < b.start; });
        rejected += !used;
    }
    h_info[0] = total; h_info[2] = rejected; h_info[3] = rounds; h_info[4] = serial;
    h_info[5] = (int64_t)links.size(); h_info[6] = longest_later;
    const Link &last = links.back();
    if ((last.end + 7) / 8 != payload_bytes) return data_error(PHM_INFLATE_TRAILING, last.start);
    if ((uint32_t)total != isize) return data_error(PHM_INFLATE_ISIZE, last.start);
    const Header h = {(int64_t)links.size(), total, payload_bytes, n};
    PHM_CUDA_CHECK(cudaMemcpyAsync(ws.links, links.data(), links.size() * sizeof(Link), cudaMemcpyHostToDevice, st));
    PHM_CUDA_CHECK(cudaMemcpyAsync(ws.hdr, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    return PHM_OK;
}

extern "C" int phm_gunzip_extract(const uint8_t *d_payload, int64_t payload_bytes, uint32_t crc32, void *d_index_workspace,
                                  size_t index_workspace_bytes, uint8_t *d_out, int64_t out_bytes, void *d_workspace, size_t workspace_bytes,
                                  void *stream) {
    PHM_REQUIRE(payload_bytes >= 0 && out_bytes >= 0, "negative size");
    PHM_REQUIRE(d_payload != nullptr || payload_bytes == 0, "d_payload is null");
    PHM_REQUIRE(d_out != nullptr || out_bytes == 0, "d_out is null");
    PHM_REQUIRE(((uintptr_t)d_out & 15u) == 0, "d_out must be 16-byte aligned");
    PHM_REQUIRE(d_index_workspace != nullptr && d_workspace != nullptr, "null pointer");
    PHM_REQUIRE(index_workspace_bytes >= 256, "index workspace too small");
    const size_t need = phm_gunzip_extract_workspace_bytes(out_bytes);
    if (workspace_bytes < need) { set_error("workspace too small: %zu < %zu", workspace_bytes, need); return PHM_E_WORKSPACE; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Header h;
    PHM_CUDA_CHECK(cudaMemcpyAsync(&h, d_index_workspace, sizeof(h), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h.payload_bytes != payload_bytes || h.total != out_bytes || h.n_links < 1 || h.n_links > h.n_chunks) {
        set_error("invalid argument: the index workspace describes %lld payload and %lld output bytes, not %lld and %lld "
                  "(call phm_gunzip_index first, on the same payload)", (long long)h.payload_bytes, (long long)h.total,
                  (long long)payload_bytes, (long long)out_bytes);
        return PHM_E_ARG;
    }
    const IndexLayout ws(d_index_workspace, h.n_chunks);
    PHM_REQUIRE(index_workspace_bytes >= ws.bytes, "index workspace too small");
    unsigned char *base = static_cast<unsigned char *>(d_workspace);
    unsigned long long *d_first = reinterpret_cast<unsigned long long *>(base);
    uint32_t *d_crc = reinterpret_cast<uint32_t *>(base + 8);
    uint16_t *d_sym = reinterpret_cast<uint16_t *>(base + 256);
    PHM_CUDA_CHECK(cudaMemsetAsync(d_first, 0xFF, sizeof(unsigned long long), st));
    PHM_CUDA_CHECK(cudaMemsetAsync(d_crc, 0, sizeof(uint32_t), st));
    gunzip_symbol_kernel<<<grid_for(h.n_links, WARPS), WARPS * 32, 0, st>>>(d_payload, payload_bytes, ws.links, h.n_links, d_sym, d_first);
    PHM_LAUNCH_CHECK();
    // Pass C reads only what pass B wrote: a failed link (a match before the stream's start, say, which pass A cannot see past
    // the first link) leaves part of its symbol range as the workspace held it, so the call stops here.
    unsigned long long first = 0;
    PHM_CUDA_CHECK(cudaMemcpyAsync(&first, d_first, sizeof(first), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (first != ~0ull) {
        set_error("corrupt DEFLATE data: piece %lld: %s (status %d)", (long long)(first >> 8), gunzip_reason((int)(first & 255ull)),
                  (int)(first & 255ull));
        return PHM_E_DATA;
    }
    if (out_bytes > 0) {
        gunzip_literal_kernel<<<grid_for(out_bytes / 8 + 1, 256), 256, 0, st>>>(d_sym, out_bytes, d_out);
        PHM_LAUNCH_CHECK();
        gunzip_tail_kernel<<<1, RESOLVE_THREADS, 0, st>>>(ws.links, h.n_links, d_sym, d_out);
        PHM_LAUNCH_CHECK();
        gunzip_marker_kernel<<<grid_for(out_bytes / 8 + 1, 256), 256, 0, st>>>(ws.links, h.n_links, d_sym, out_bytes, d_out);
        PHM_LAUNCH_CHECK();
        const int threads = 256, blocks = sm_count() * 8;
        const int64_t pieces = (int64_t)threads * blocks;
        const int64_t piece = ((out_bytes + pieces - 1) / pieces + 15) / 16 * 16;
        gunzip_crc_kernel<<<blocks, threads, 0, st>>>(d_out, out_bytes, piece, d_crc);
        PHM_LAUNCH_CHECK();
    }
    uint32_t crc = 0;
    PHM_CUDA_CHECK(cudaMemcpyAsync(&crc, d_crc, sizeof(crc), cudaMemcpyDeviceToHost, st));
    PHM_CUDA_CHECK(cudaStreamSynchronize(st));
    if (crc != crc32) return data_error(PHM_INFLATE_CRC, 0);
    return PHM_OK;
}
