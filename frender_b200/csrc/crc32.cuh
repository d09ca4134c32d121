// CRC-32 (RFC 1952) on the device, shared by the inflate check (gz_kernels.cuh) and the encoder
// (deflate_kernels.cuh).  Standard CRC-32 values combine like zlib's crc32_combine:
// crc(A || B) = x^(8 |B|) * crc(A) + crc(B) in GF(2)[x] / P (reflected bit order, bit 31 = x^0), so pieces of a
// text are summed independently and joined.
#pragma once
#include <cuda_runtime.h>

namespace frb {
namespace gz {

// x^(2^k) mod P for k < 32 (P = the CRC-32 polynomial, reflected; made by the host), kernel parameter
struct CrcPowers {
    unsigned int x2n[32];
};

constexpr unsigned kCrcPoly = 0xEDB88320u;

__device__ __forceinline__ unsigned crc_mul(unsigned a, unsigned b) {  // a * b mod P
    unsigned p = 0;
#pragma unroll 4
    for (int k = 0; k < 32; ++k) {
        p ^= b & (0u - ((a >> (31 - k)) & 1u));
        b = (b >> 1) ^ (kCrcPoly & (0u - (b & 1u)));
    }
    return p;
}
__device__ inline unsigned crc_xpow8(const CrcPowers& pw, unsigned long long nbytes) {  // x^(8 nbytes) mod P
    unsigned p = 0x80000000u;
    for (int k = 3; nbytes; nbytes >>= 1, ++k)
        if (nbytes & 1) p = crc_mul(pw.x2n[k & 31], p);
    return p;
}
__device__ __forceinline__ unsigned crc_join(const CrcPowers& pw, unsigned crc_a, unsigned crc_b, unsigned long long len_b) {
    return len_b ? (crc_mul(crc_xpow8(pw, len_b), crc_a) ^ crc_b) : crc_a;
}
__device__ inline unsigned crc_bytes(const unsigned char* __restrict__ p, unsigned n) {  // crc32 of n bytes, bit by bit
    unsigned crc = 0xFFFFFFFFu;
    for (unsigned i = 0; i < n; ++i) {
        crc ^= p[i];
#pragma unroll
        for (int k = 0; k < 8; ++k) crc = (crc >> 1) ^ (kCrcPoly & (0u - (crc & 1u)));
    }
    return ~crc;
}

}  // namespace gz
}  // namespace frb
