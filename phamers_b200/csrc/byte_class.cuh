// SWAR byte classes shared by the text scanners (fasta_scan.cu, feature_csv.cu): four bytes of a 32-bit word tested at once, and
// the per-byte results gathered into a 4-bit mask.
#pragma once
#include <stdint.h>

namespace phm {

// 0x80 in every byte of x that is zero
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
    return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
}
// bits 7, 15, 23, 31 -> bits 0..3 (the partial products land on distinct bits, so there are no carries)
__device__ __forceinline__ uint32_t gather4(uint32_t z) { return (((z >> 7) * 0x00204081u) >> 21) & 0xFu; }

}  // namespace phm
