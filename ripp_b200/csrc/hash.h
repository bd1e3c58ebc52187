// Host-side hashes for the Fiat-Shamir transcripts: BLAKE2b-512 (GIPA/TIPA/aggregation challenges,
// gipa.rs:235-258, tipa/mod.rs:195-209, groth16_aggregation.rs:105-116), BLAKE2s-256 and the
// ChaCha20 block function (SIPP's hash-reseeded RNG, sipp/src/rng.rs:12-73; also called on the device for the
// scalars of the Groth16 random-linear-combination check, groth16.cu).  RFC 7693 / RFC 8439,
// unkeyed, written from the RFCs.
#pragma once
#include <stdint.h>
#include <string.h>

#include <vector>

#ifndef RIPP_HD  // as limb.cuh defines it
#if defined(__CUDACC__)
#define RIPP_HD __host__ __device__ __forceinline__
#else
#define RIPP_HD inline
#endif
#endif

namespace ripp_hash {

static inline uint64_t rotr64(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
static inline uint32_t rotr32(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
RIPP_HD uint32_t rotl32(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }

static const uint8_t SIGMA[12][16] = {
    {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
    {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
    {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
    {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
    {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0},
    {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3}};

static const uint64_t IV64[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                                 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
static const uint32_t IV32[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au,
                                 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};

static inline void b2b_compress(uint64_t h[8], const uint8_t block[128], uint64_t t, bool last) {
  uint64_t m[16], v[16];
  memcpy(m, block, 128);
  for (int i = 0; i < 8; i++) {
    v[i] = h[i];
    v[i + 8] = IV64[i];
  }
  v[12] ^= t;
  if (last) v[14] = ~v[14];
#define G(a, b, c, d, x, y)      \
  v[a] = v[a] + v[b] + x;        \
  v[d] = rotr64(v[d] ^ v[a], 32); \
  v[c] = v[c] + v[d];            \
  v[b] = rotr64(v[b] ^ v[c], 24); \
  v[a] = v[a] + v[b] + y;        \
  v[d] = rotr64(v[d] ^ v[a], 16); \
  v[c] = v[c] + v[d];            \
  v[b] = rotr64(v[b] ^ v[c], 63);
  for (int r = 0; r < 12; r++) {
    const uint8_t* s = SIGMA[r];
    G(0, 4, 8, 12, m[s[0]], m[s[1]]) G(1, 5, 9, 13, m[s[2]], m[s[3]]) G(2, 6, 10, 14, m[s[4]], m[s[5]])
        G(3, 7, 11, 15, m[s[6]], m[s[7]]) G(0, 5, 10, 15, m[s[8]], m[s[9]]) G(1, 6, 11, 12, m[s[10]], m[s[11]])
            G(2, 7, 8, 13, m[s[12]], m[s[13]]) G(3, 4, 9, 14, m[s[14]], m[s[15]])
  }
#undef G
  for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
}

// BLAKE2b with 64-byte digest, no key
static inline void blake2b512(const uint8_t* data, size_t len, uint8_t out[64]) {
  uint64_t h[8];
  for (int i = 0; i < 8; i++) h[i] = IV64[i];
  h[0] ^= 0x01010000ull ^ 64ull;
  uint8_t block[128];
  size_t off = 0;
  while (len - off > 128) {
    b2b_compress(h, data + off, off + 128, false);
    off += 128;
  }
  memset(block, 0, 128);
  memcpy(block, data + off, len - off);
  b2b_compress(h, block, len, true);
  memcpy(out, h, 64);
}

static inline void b2s_compress(uint32_t h[8], const uint8_t block[64], uint64_t t, bool last) {
  uint32_t m[16], v[16];
  memcpy(m, block, 64);
  for (int i = 0; i < 8; i++) {
    v[i] = h[i];
    v[i + 8] = IV32[i];
  }
  v[12] ^= (uint32_t)t;
  v[13] ^= (uint32_t)(t >> 32);
  if (last) v[14] = ~v[14];
#define G(a, b, c, d, x, y)      \
  v[a] = v[a] + v[b] + x;        \
  v[d] = rotr32(v[d] ^ v[a], 16); \
  v[c] = v[c] + v[d];            \
  v[b] = rotr32(v[b] ^ v[c], 12); \
  v[a] = v[a] + v[b] + y;        \
  v[d] = rotr32(v[d] ^ v[a], 8);  \
  v[c] = v[c] + v[d];            \
  v[b] = rotr32(v[b] ^ v[c], 7);
  for (int r = 0; r < 10; r++) {
    const uint8_t* s = SIGMA[r];
    G(0, 4, 8, 12, m[s[0]], m[s[1]]) G(1, 5, 9, 13, m[s[2]], m[s[3]]) G(2, 6, 10, 14, m[s[4]], m[s[5]])
        G(3, 7, 11, 15, m[s[6]], m[s[7]]) G(0, 5, 10, 15, m[s[8]], m[s[9]]) G(1, 6, 11, 12, m[s[10]], m[s[11]])
            G(2, 7, 8, 13, m[s[12]], m[s[13]]) G(3, 4, 9, 14, m[s[14]], m[s[15]])
  }
#undef G
  for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
}

// BLAKE2s with 32-byte digest, no key
static inline void blake2s256(const uint8_t* data, size_t len, uint8_t out[32]) {
  uint32_t h[8];
  for (int i = 0; i < 8; i++) h[i] = IV32[i];
  h[0] ^= 0x01010000u ^ 32u;
  uint8_t block[64];
  size_t off = 0;
  while (len - off > 64) {
    b2s_compress(h, data + off, off + 64, false);
    off += 64;
  }
  memset(block, 0, 64);
  memcpy(block, data + off, len - off);
  b2s_compress(h, block, len, true);
  memcpy(out, h, 32);
}

// ChaCha20 block (rand_chacha 0.3 ChaChaRng: 64-bit block counter in words 12-13, stream 0)
RIPP_HD void chacha20_block(const uint8_t key[32], uint64_t counter, uint8_t out[64]) {
  uint32_t init[16], s[16];
  init[0] = 0x61707865u;  // "expand 32-byte k"
  init[1] = 0x3320646eu;
  init[2] = 0x79622d32u;
  init[3] = 0x6b206574u;
  memcpy(init + 4, key, 32);
  init[12] = (uint32_t)counter;
  init[13] = (uint32_t)(counter >> 32);
  init[14] = init[15] = 0;
  memcpy(s, init, 64);
#define QR(a, b, c, d)            \
  s[a] += s[b];                   \
  s[d] = rotl32(s[d] ^ s[a], 16); \
  s[c] += s[d];                   \
  s[b] = rotl32(s[b] ^ s[c], 12); \
  s[a] += s[b];                   \
  s[d] = rotl32(s[d] ^ s[a], 8);  \
  s[c] += s[d];                   \
  s[b] = rotl32(s[b] ^ s[c], 7);
  for (int i = 0; i < 10; i++) {
    QR(0, 4, 8, 12) QR(1, 5, 9, 13) QR(2, 6, 10, 14) QR(3, 7, 11, 15) QR(0, 5, 10, 15) QR(1, 6, 11, 12) QR(2, 7, 8, 13)
        QR(3, 4, 9, 14)
  }
#undef QR
  for (int i = 0; i < 16; i++) s[i] += init[i];
  memcpy(out, s, 64);
}

}  // namespace ripp_hash
