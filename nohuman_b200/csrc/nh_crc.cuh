/* nh_crc.cuh — CRC-32 (gzip's reflected polynomial 0xedb88320) algebra shared by the deflate and inflate
 * kernels: a CRC computed over a slice moves past the n bytes that follow it by a multiplication with
 * x^(8n) mod P, so slices computed in parallel XOR together (zlib's crc32_combine). */
#ifndef NH_CRC_CUH
#define NH_CRC_CUH

#include <stdint.h>

namespace {

/* x^(2^k) mod P for the reflected CRC-32 polynomial (zlib's x2n_table) */
__constant__ uint32_t c_x2n[32] = {
    0x40000000, 0x20000000, 0x08000000, 0x00800000, 0x00008000, 0xedb88320, 0xb1e6b092, 0xa06a2517,
    0xed627dae, 0x88d14467, 0xd7bbfe6a, 0xec447f11, 0x8e7ea170, 0x6427800e, 0x4d47bae0, 0x09fe548f,
    0x83852d0f, 0x30362f1a, 0x7b5a9cc3, 0x31fec169, 0x9fec022a, 0x6c8dedc4, 0x15d6874d, 0x5fde7a4e,
    0xbad90e37, 0x2e4e5eef, 0x4eaba214, 0xa8a472c0, 0x429a969e, 0x148d302a, 0xc40ba6d0, 0xc4e22c3c};

/* a(x) * b(x) mod P, reflected */
__device__ uint32_t crc_mulmod(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
  }
  return p;
}

/* x^(8 n) mod P: the factor that moves a CRC past n zero bytes */
__device__ uint32_t crc_x8n(uint64_t n) {
  uint32_t p = 1u << 31;
  for (int k = 3; n; n >>= 1, k++)
    if (n & 1) p = crc_mulmod(c_x2n[k & 31], p);
  return p;
}

}  // namespace

#endif
