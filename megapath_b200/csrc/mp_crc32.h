// mp_crc32.h -- CRC-32 (gzip polynomial, reflected) arithmetic shared by the BGZF encoder and the gzip decoder, host and device:
// the product of two polynomials mod P and x^(8n) mod P, from which crc32_combine follows (zlib crc32.c).
#pragma once
#include <stdint.h>

__host__ __device__ __forceinline__ uint32_t mp_crc32_mulmod(uint32_t a, uint32_t b)      // a * b mod P, reflected
{
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
__host__ __device__ inline uint32_t mp_crc32_x8n(uint64_t n)                                 // x^(8n) mod P
{
    uint32_t p = 1u << 31, sq = 1u << 30;                                                     // sq = x^(2^k) while k walks up from 0
    for (int k = 0; k < 3; ++k) sq = mp_crc32_mulmod(sq, sq);                                  // x^8
    while (n) {
        if (n & 1) p = mp_crc32_mulmod(sq, p);
        n >>= 1;
        if (n) sq = mp_crc32_mulmod(sq, sq);
    }
    return p;
}
// CRC-32 of A followed by B from crc(A), crc(B) and |B| (zlib's crc32_combine)
__host__ __device__ inline uint32_t mp_crc32_combine(uint32_t crcA, uint32_t crcB, uint64_t lenB)
{
    return mp_crc32_mulmod(mp_crc32_x8n(lenB), crcA) ^ crcB;
}
