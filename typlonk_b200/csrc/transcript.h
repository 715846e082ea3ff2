// Host-side Fiat-Shamir of the prover: restates plonk/src/proof/challenges.rs:9-46 --
// transcript = ark-serialize 0.3 `serialize_unchecked` of each G1 commitment (96 B: x, y as
// little-endian canonical integers, flag bits in the top of the last byte), Blake2b-512, first
// 8 bytes LE as seed, rand 0.8 `StdRng::seed_from_u64` (PCG32 expansion -> ChaCha12) and
// ark-ff 0.3 `Fr::rand` (4 x u64, top bit cleared, rejection-sampled, taken AS the Montgomery
// representation).  Product code (independent of oracle/); negligible cost, but it decides
// every later byte of the proof.
#pragma once
#include <stdint.h>
#include <string.h>
#include <vector>

#include "host_field.h"

namespace tph {

// ---- Blake2b-512 (RFC 7693), unkeyed --------------------------------------------------
struct Blake2b {
  uint64_t h[8];
  uint64_t t[2];
  uint8_t buf[128];
  size_t buflen;

  static uint64_t rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
  static uint64_t load64(const uint8_t* p) {
    uint64_t v = 0;
    for (int i = 7; i >= 0; i--) v = (v << 8) | p[i];
    return v;
  }
  void init() {
    static const uint64_t iv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull,
                                   0xa54ff53a5f1d36f1ull, 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full,
                                   0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    memcpy(h, iv, sizeof(h));
    h[0] ^= 0x01010000ull ^ 64;  // digest length 64, no key, fanout = depth = 1
    t[0] = t[1] = 0;
    buflen = 0;
  }
  void compress(const uint8_t* block, bool last) {
    static const uint64_t iv[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull,
                                   0xa54ff53a5f1d36f1ull, 0x510e527fade682d1ull, 0x9b05688c2b3e6c1full,
                                   0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    static const uint8_t sigma[12][16] = {
        {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
        {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
        {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
        {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
        {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0},
        {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3}};
    uint64_t m[16], v[16];
    for (int i = 0; i < 16; i++) m[i] = load64(block + 8 * i);
    for (int i = 0; i < 8; i++) {
      v[i] = h[i];
      v[i + 8] = iv[i];
    }
    v[12] ^= t[0];
    v[13] ^= t[1];
    if (last) v[14] = ~v[14];
#define TP_B2G(a, b, c, d, x, y)        \
  v[a] = v[a] + v[b] + (x);             \
  v[d] = rotr(v[d] ^ v[a], 32);         \
  v[c] = v[c] + v[d];                   \
  v[b] = rotr(v[b] ^ v[c], 24);         \
  v[a] = v[a] + v[b] + (y);             \
  v[d] = rotr(v[d] ^ v[a], 16);         \
  v[c] = v[c] + v[d];                   \
  v[b] = rotr(v[b] ^ v[c], 63);
    for (int r = 0; r < 12; r++) {
      const uint8_t* s = sigma[r];
      TP_B2G(0, 4, 8, 12, m[s[0]], m[s[1]]);
      TP_B2G(1, 5, 9, 13, m[s[2]], m[s[3]]);
      TP_B2G(2, 6, 10, 14, m[s[4]], m[s[5]]);
      TP_B2G(3, 7, 11, 15, m[s[6]], m[s[7]]);
      TP_B2G(0, 5, 10, 15, m[s[8]], m[s[9]]);
      TP_B2G(1, 6, 11, 12, m[s[10]], m[s[11]]);
      TP_B2G(2, 7, 8, 13, m[s[12]], m[s[13]]);
      TP_B2G(3, 4, 9, 14, m[s[14]], m[s[15]]);
    }
#undef TP_B2G
    for (int i = 0; i < 8; i++) h[i] ^= v[i] ^ v[i + 8];
  }
  void update(const uint8_t* in, size_t len) {
    while (len > 0) {
      if (buflen == 128) {
        t[0] += 128;
        if (t[0] < 128) t[1]++;
        compress(buf, false);
        buflen = 0;
      }
      size_t take = 128 - buflen < len ? 128 - buflen : len;
      memcpy(buf + buflen, in, take);
      buflen += take;
      in += take;
      len -= take;
    }
  }
  void finalize(uint8_t out[64]) {
    t[0] += buflen;
    if (t[0] < buflen) t[1]++;
    memset(buf + buflen, 0, 128 - buflen);
    compress(buf, true);
    for (int i = 0; i < 8; i++)
      for (int j = 0; j < 8; j++) out[8 * i + j] = (uint8_t)(h[i] >> (8 * j));
  }
};

// ---- ChaCha12 StdRng -------------------------------------------------------------------
struct StdRng {
  uint32_t key[8];
  uint64_t counter;
  uint32_t block[16];
  int pos;

  static uint32_t rotl(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }
  static StdRng seed_from_u64(uint64_t state) {
    StdRng r;
    const uint64_t MUL = 6364136223846793005ull, INC = 11634580027462260723ull;
    for (int i = 0; i < 8; i++) {
      state = state * MUL + INC;
      uint32_t xorshifted = (uint32_t)(((state >> 18) ^ state) >> 27);
      uint32_t rot = (uint32_t)(state >> 59);
      r.key[i] = (xorshifted >> rot) | (xorshifted << ((32 - rot) & 31));
    }
    r.counter = 0;
    r.pos = 16;
    return r;
  }
  // `SeedableRng::from_seed`: the 32 bytes are the ChaCha key, little-endian words
  static StdRng from_seed(const uint8_t seed[32]) {
    StdRng r;
    for (int i = 0; i < 8; i++)
      r.key[i] = (uint32_t)seed[4 * i] | ((uint32_t)seed[4 * i + 1] << 8) | ((uint32_t)seed[4 * i + 2] << 16) | ((uint32_t)seed[4 * i + 3] << 24);
    r.counter = 0;
    r.pos = 16;
    return r;
  }
  void refill() {
    uint32_t init[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u};
    for (int i = 0; i < 8; i++) init[4 + i] = key[i];
    init[12] = (uint32_t)counter;
    init[13] = (uint32_t)(counter >> 32);
    init[14] = init[15] = 0;
    uint32_t s[16];
    memcpy(s, init, sizeof(s));
#define TP_QR(a, b, c, d)                 \
  s[a] += s[b]; s[d] = rotl(s[d] ^ s[a], 16); \
  s[c] += s[d]; s[b] = rotl(s[b] ^ s[c], 12); \
  s[a] += s[b]; s[d] = rotl(s[d] ^ s[a], 8);  \
  s[c] += s[d]; s[b] = rotl(s[b] ^ s[c], 7);
    for (int r = 0; r < 6; r++) {
      TP_QR(0, 4, 8, 12) TP_QR(1, 5, 9, 13) TP_QR(2, 6, 10, 14) TP_QR(3, 7, 11, 15)
      TP_QR(0, 5, 10, 15) TP_QR(1, 6, 11, 12) TP_QR(2, 7, 8, 13) TP_QR(3, 4, 9, 14)
    }
#undef TP_QR
    for (int i = 0; i < 16; i++) block[i] = s[i] + init[i];
    counter++;
    pos = 0;
  }
  uint32_t next_u32() {
    if (pos >= 16) refill();
    return block[pos++];
  }
  uint64_t next_u64() {
    uint64_t lo = next_u32();
    uint64_t hi = next_u32();
    return lo | (hi << 32);
  }
};

// ark-ff 0.3 Fr::rand: accepted limbs ARE the Montgomery representation.
static inline HFr fr_rand(StdRng& rng) {
  for (;;) {
    HFr r;
    for (int i = 0; i < 4; i++) r.v[i] = rng.next_u64();
    r.v[3] &= 0xffffffffffffffffull >> 1;
    if (!ge<4>(r.v, FR_PARAMS.mod)) return r;
  }
}

// ark-serialize 0.3 uncompressed G1 (96 B) from the 97-byte ABI point (Montgomery x | y | inf).
static inline void serialize_g1_unchecked(const uint8_t pt[97], uint8_t out[96]) {
  if (pt[96]) {
    memset(out, 0, 96);
    out[48] = 1;          // y = 1
    out[95] |= 1 << 6;    // SWFlags::Infinity
    return;
  }
  HFq x, y;
  memcpy(x.v, pt, 48);
  memcpy(y.v, pt + 48, 48);
  HFq xc = x.from_mont(), yc = y.from_mont();
  memcpy(out, xc.v, 48);
  memcpy(out + 48, yc.v, 48);
}

// ChallengeGenerator::generate_challenges::<2>() over the given commitments.
static inline void challenges2(const std::vector<const uint8_t*>& commitments, HFr* c0, HFr* c1) {
  Blake2b b;
  b.init();
  for (const uint8_t* p : commitments) {
    uint8_t ser[96];
    serialize_g1_unchecked(p, ser);
    b.update(ser, 96);
  }
  uint8_t digest[64];
  b.finalize(digest);
  uint64_t seed = 0;
  for (int i = 7; i >= 0; i--) seed = (seed << 8) | digest[i];
  StdRng rng = StdRng::seed_from_u64(seed);
  *c0 = fr_rand(rng);
  *c1 = fr_rand(rng);
}

// Proof format v2 (DESIGN.md, "Proof format v2"): H = Blake2b-512, s = H("typlonk-plonk-v2" | H(key bytes) | u64 LE l
// | public values), absorb: s = H(s | label | data), squeeze(i) = LE-int(H(s | "challenge" | u8 i)) mod r.
// G1 as serialize_g1_unchecked (96 B), Fr as 32 B canonical LE.
struct TranscriptV2 {
  uint8_t s[64];

  static void put_fr(Blake2b& b, const HFr& x) {
    HFr c = x.from_mont();
    b.update((const uint8_t*)c.v, 32);
  }
  void init(const uint8_t vk_digest[64], const HFr* publics, size_t count) {
    Blake2b b;
    b.init();
    b.update((const uint8_t*)"typlonk-plonk-v2", 16);
    b.update(vk_digest, 64);
    uint8_t l[8];
    for (int i = 0; i < 8; i++) l[i] = (uint8_t)((uint64_t)count >> (8 * i));
    b.update(l, 8);
    for (size_t i = 0; i < count; i++) put_fr(b, publics[i]);
    b.finalize(s);
  }
  // points: 97-byte ABI records
  void absorb(const char* label, const std::vector<const uint8_t*>& points, const HFr* frs = nullptr, int nfr = 0) {
    Blake2b b;
    b.init();
    b.update(s, 64);
    b.update((const uint8_t*)label, strlen(label));
    for (const uint8_t* p : points) {
      uint8_t ser[96];
      serialize_g1_unchecked(p, ser);
      b.update(ser, 96);
    }
    for (int i = 0; i < nfr; i++) put_fr(b, frs[i]);
    b.finalize(s);
  }
  HFr squeeze(uint8_t i) const {
    Blake2b b;
    b.init();
    b.update(s, 64);
    b.update((const uint8_t*)"challenge", 9);
    b.update(&i, 1);
    uint8_t d[64];
    b.finalize(d);
    // 512-bit little-endian integer mod r, Horner over 64-bit limbs from the top
    const HFr two32 = HFr::from_u64((uint64_t)1 << 32), two64 = two32 * two32;
    HFr acc = HFr::zero();
    for (int k = 7; k >= 0; k--) {
      uint64_t limb = 0;
      for (int j = 7; j >= 0; j--) limb = (limb << 8) | d[8 * k + j];
      acc = acc * two64 + HFr::from_u64(limb);
    }
    return acc;
  }
};

}  // namespace tph
