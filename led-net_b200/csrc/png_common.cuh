// CRC-32 (PNG chunks) and Adler-32 (zlib streams), shared by the PNG encoder (png.cu) and decoder (png_decode.cu).
// Everything here is __host__ __device__: the decoder's diagnostic host entry point runs the same code on the CPU.
#pragma once
#include <stdint.h>

namespace ledb {

constexpr uint32_t kCrcPoly = 0xedb88320u;
constexpr uint32_t kAdlerMod = 65521;

// entry t of the byte-wise CRC-32 table
__host__ __device__ inline uint32_t crc_table_entry(uint32_t t) {
  for (int k = 0; k < 8; ++k) t = (t & 1) ? (t >> 1) ^ kCrcPoly : t >> 1;
  return t;
}

// the running (un-inverted) CRC register c advanced over p[0, n)
__host__ __device__ inline uint32_t crc_update(const uint32_t* tab, uint32_t c, const uint8_t* p, int64_t n) {
  for (int64_t i = 0; i < n; ++i) c = tab[(c ^ p[i]) & 0xff] ^ (c >> 8);
  return c;
}

// a * b modulo the CRC-32 polynomial, bit-reflected (zlib's multmodp)
__host__ __device__ inline uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, r = 0;
  for (;;) {
    if (a & m) {
      r ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return r;
}

// x2n[k] = x^(2^k) mod P, k < 32
__host__ __device__ inline void crc_x2n_table(uint32_t* x2n) {
  x2n[0] = 1u << 30;                            // x^1
  for (int k = 1; k < 32; ++k) x2n[k] = crc_multmodp(x2n[k - 1], x2n[k - 1]);
}

// crc32(A || B) from crc32(A), crc32(B) and |B|
__host__ __device__ inline uint32_t crc_combine(uint32_t c1, uint32_t c2, int64_t len2, const uint32_t* x2n) {
  uint32_t pw = 1u << 31;                       // x^0
  int k = 3;                                    // x^(8 len2): start at 2^3
  for (int64_t n = len2; n; n >>= 1, ++k)
    if (n & 1) pw = crc_multmodp(x2n[k & 31], pw);
  return crc_multmodp(pw, c1) ^ c2;
}

// Adler-32 sums of a segment p[0, n): s1 = sum of the bytes, s2 = sum of the running s1 (= sum of (n - i) p[i]), both
// mod 65521.  Segments combine by addition once s2 is shifted by the bytes after the segment (adler_shift).
__host__ __device__ inline void adler_sums(const uint8_t* p, int64_t n, uint64_t& s1, uint64_t& s2) {
  s1 = 0; s2 = 0;
  for (int64_t i0 = 0; i0 < n; i0 += 5552) {    // reduced every 5552 bytes (zlib's NMAX)
    const int64_t i1 = n - i0 < 5552 ? n : i0 + 5552;
    for (int64_t i = i0; i < i1; ++i) { s1 += p[i]; s2 += s1; }
    s1 %= kAdlerMod; s2 %= kAdlerMod;
  }
}
// s2 of a segment followed by `rest` more bytes
__host__ __device__ inline uint64_t adler_shift(uint64_t s1, uint64_t s2, int64_t rest) {
  return (s2 + s1 * ((uint64_t)rest % kAdlerMod)) % kAdlerMod;
}
// the Adler-32 of an n-byte stream whose segment sums add up to (s1, s2)
__host__ __device__ inline uint32_t adler_final(uint64_t s1, uint64_t s2, int64_t n) {
  return (uint32_t)((((uint64_t)n % kAdlerMod + s2) % kAdlerMod) << 16 | (1 + s1) % kAdlerMod);
}

}  // namespace ledb
