// Wire formats (SURVEY.md 8 f4, App. A.6): a proof and an SRS as bytes, in the encoding ark-serialize 0.3 gives the
// reference's own types -- the same one its Fiat-Shamir transcript already uses for G1 (plonk/src/proof/challenges.rs:17-22):
//   Fr  32 B little-endian canonical integer
//   G1  96 B uncompressed: x | y, 48 B little-endian canonical each; bit 6 of the last byte = point at infinity
//       (stored as x = 0, y = 1); bit 7 is the y-sign flag of the COMPRESSED form and must be clear here
//   G2  192 B uncompressed: x.c0 | x.c1 | y.c0 | y.c1, same flag convention
//   Vec u64 little-endian length, then the items
// Proof (plonk/src/proof.rs:85-95)  = the 1472-byte block tp_prove writes | Vec<Fr> public inputs.
// SRS   (kzg/src/srs.rs:8-14)       = Vec<G1> | G2 | tau G2.
// The reference derives neither Serialize nor Deserialize for these types, so the framing is ours; every item inside
// it is what arkworks would write.  Proofs are small and handled on the host; the SRS (100 MB at 2^20) is converted
// out of / into Montgomery form and validated (canonical, on the curve, optionally in the prime-order subgroup) on
// the device, one point per thread.
// Both also exist with compressed points (ark `serialize`): G1 = x with the y-sign flag (48 B), G2 = x.c0 | x.c1 with
// the flags in x.c1 (96 B).  Decompression costs one square root per point: on the device for the SRS and for batches
// of proofs (tp_proofs_decompress), on the host for single proofs and the two G2 points.
#include "circuit.h"
#include "ec.cuh"
#include "pairing.h"

using namespace tp;
using namespace tph;

namespace tp {

__device__ __forceinline__ bool fq_lt_mod(const Fq& a) {
  const uint32_t m[12] = TP_FQ_MOD;
  for (int i = 11; i >= 0; i--) {
    if (a.v[i] < m[i]) return true;
    if (a.v[i] > m[i]) return false;
  }
  return false;
}
__device__ __forceinline__ Fq fq_to_mont(const Fq& a) {
  const uint32_t c[12] = TP_FQ_R2;
  Fq r2;
#pragma unroll
  for (int i = 0; i < 12; i++) r2.v[i] = c[i];
  return fq_mul(a, r2);
}
__device__ __forceinline__ Fq fq_from_mont(const Fq& a) {
  Fq o = fq_zero();
  o.v[0] = 1;
  return fq_mul(a, o);
}

// Montgomery SRS records -> wire records.  96 B per thread as six 16-byte stores.
__global__ void __launch_bounds__(128) k_g1_to_wire(const G1Affine* __restrict__ in, size_t len, uint4* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    G1Affine p = affine_load(in + i);
    Fq x, y;
    if (affine_is_identity(p)) {
      x = fq_zero();
      y = fq_zero();
      y.v[0] = 1;
      y.v[11] |= 0x40000000u;  // bit 6 of byte 95
    } else {
      x = fq_from_mont(p.x);
      y = fq_from_mont(p.y);
    }
    uint4* o = out + i * 6;
    o[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    o[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
    o[2] = make_uint4(x.v[8], x.v[9], x.v[10], x.v[11]);
    o[3] = make_uint4(y.v[0], y.v[1], y.v[2], y.v[3]);
    o[4] = make_uint4(y.v[4], y.v[5], y.v[6], y.v[7]);
    o[5] = make_uint4(y.v[8], y.v[9], y.v[10], y.v[11]);
  }
}

// Wire records -> Montgomery SRS records, validated.  check: 0 = canonical encoding only (deserialize_unchecked),
// 1 = + on the curve, 2 = + in the prime-order subgroup (what ark-ec's checked deserialisation enforces).
// bad[0] counts rejected records, bad[1] keeps the lowest rejected index + 1.
__global__ void __launch_bounds__(128) k_g1_from_wire(const uint4* __restrict__ in, size_t len, int check,
                                                      G1Affine* __restrict__ out, unsigned long long* __restrict__ bad) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    const uint4* s = in + i * 6;
    Fq x, y;
    uint4 q;
    q = s[0]; x.v[0] = q.x; x.v[1] = q.y; x.v[2] = q.z; x.v[3] = q.w;
    q = s[1]; x.v[4] = q.x; x.v[5] = q.y; x.v[6] = q.z; x.v[7] = q.w;
    q = s[2]; x.v[8] = q.x; x.v[9] = q.y; x.v[10] = q.z; x.v[11] = q.w;
    q = s[3]; y.v[0] = q.x; y.v[1] = q.y; y.v[2] = q.z; y.v[3] = q.w;
    q = s[4]; y.v[4] = q.x; y.v[5] = q.y; y.v[6] = q.z; y.v[7] = q.w;
    q = s[5]; y.v[8] = q.x; y.v[9] = q.y; y.v[10] = q.z; y.v[11] = q.w;
    const uint32_t flags = y.v[11] >> 30;
    y.v[11] &= 0x3fffffffu;
    bool ok = !(flags & 2) && fq_lt_mod(x) && fq_lt_mod(y);
    G1Affine p;
    if (flags & 1) {  // infinity: canonical only as (x, y) = (0, 1); the device SRS keeps it as the all-zero record
      bool canon = x.v[0] == 0 && y.v[0] == 1;
#pragma unroll
      for (int k = 1; k < 12; k++) canon = canon && x.v[k] == 0 && y.v[k] == 0;
      ok = ok && canon;
      p.x = fq_zero();
      p.y = fq_zero();
    } else {
      p.x = fq_to_mont(x);
      p.y = fq_to_mont(y);
      if (ok && check >= 1) {
        Fq four = fq_dbl(fq_dbl(fq_one()));
        ok = fq_eq(fq_sqr(p.y), fq_add(fq_mul(fq_sqr(p.x), p.x), four));
      }
      if (ok && check >= 2) ok = g1_in_subgroup(p);
    }
    fq_store(&out[i].x, p.x);
    fq_store(&out[i].y, p.y);
    if (!ok) {
      atomicAdd(bad, 1ull);
      atomicMin(bad + 1, (unsigned long long)i + 1);
    }
  }
}

// ---- compressed G1 records (48 B: x | flags in the top two bits of byte 47) -----------------------------------------
// ark-ec 0.3 writes x with SWFlags: bit 7 = PositiveY (y > -y as canonical integers), bit 6 = infinity (x = 0).
// ⚠ The sign convention is recalled from the pinned crates (ark-ec 0.3 GroupAffine::serialize, `y > -y`), not checked
// against them offline; tools/arkworks_dump emits vectors that tests/test_wire_compressed.py compares when present.

// y = a^((q+1)/4), the square root of a when one exists (q = 3 mod 4).  Fixed 4-bit window over the 379-bit exponent:
// 14 products for the table a^0..a^15, 376 squarings and 91 products for the non-zero digits, 481 Fq products instead
// of 606 for square-and-multiply.  The exponent is a constant, so every lane takes the same branches.  Canonical
// (fully reduced) Fq arithmetic; the table lives in the thread's stack frame.
static __device__ __noinline__ Fq fq_pow_sqrt_exp(const Fq& a) {
  const uint32_t e[12] = TP_FQ_SQRT_EXP;
  Fq t[16];
  t[0] = fq_one();
  t[1] = a;
#pragma unroll 1
  for (int k = 2; k < 16; k++) t[k] = fq_mul(t[k - 1], a);
  Fq r = t[(e[11] >> 24) & 15];  // window 94 = bits 376..379: the top digit (bits 380..383 are zero)
#pragma unroll 1
  for (int w = 93; w >= 0; w--) {
#pragma unroll
    for (int s = 0; s < 4; s++) r = fq_sqr(r);
    const uint32_t d = (e[w >> 3] >> (4 * (w & 7))) & 15;
    if (d) r = fq_mul(r, t[d]);
  }
  return r;
}
// *y = sqrt(a) (Montgomery in, Montgomery out); false if a is not a square.
__device__ __forceinline__ bool fq_sqrt(const Fq& a, Fq* y) {
  *y = fq_pow_sqrt_exp(a);
  return fq_eq(fq_sqr(*y), a);
}
// canonical integers: a > b
__device__ __forceinline__ bool fq_gt_canon(const Fq& a, const Fq& b) {
#pragma unroll
  for (int i = 11; i >= 0; i--) {
    if (a.v[i] != b.v[i]) return a.v[i] > b.v[i];
  }
  return false;
}

// Montgomery SRS records -> compressed wire records.  48 B per thread as three 16-byte stores.
__global__ void __launch_bounds__(128) k_g1_to_wire_compressed(const G1Affine* __restrict__ in, size_t len,
                                                               uint4* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    G1Affine p = affine_load(in + i);
    Fq x;
    if (affine_is_identity(p)) {
      x = fq_zero();
      x.v[11] = 0x40000000u;  // bit 6 of byte 47
    } else {
      x = fq_from_mont(p.x);
      const Fq y = fq_from_mont(p.y);
      if (fq_gt_canon(y, fq_neg(y))) x.v[11] |= 0x80000000u;  // bit 7 of byte 47
    }
    uint4* o = out + i * 3;
    o[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    o[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
    o[2] = make_uint4(x.v[8], x.v[9], x.v[10], x.v[11]);
  }
}

// Compressed wire records -> Montgomery SRS records, validated.  check 0 and 1 both recover y (a record whose x has no
// root is rejected at every level), 2 adds [r]P = 0.  Infinity becomes the all-zero device record.  bad[] as in
// k_g1_from_wire; ok_out (may be null) gets one byte per record, 1 = accepted.
__global__ void __launch_bounds__(128) k_g1_from_wire_compressed(const uint4* __restrict__ in, size_t len, int check,
                                                                 G1Affine* __restrict__ out,
                                                                 unsigned long long* __restrict__ bad,
                                                                 uint8_t* __restrict__ ok_out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    const uint4* s = in + i * 3;
    Fq x;
    uint4 q;
    q = s[0]; x.v[0] = q.x; x.v[1] = q.y; x.v[2] = q.z; x.v[3] = q.w;
    q = s[1]; x.v[4] = q.x; x.v[5] = q.y; x.v[6] = q.z; x.v[7] = q.w;
    q = s[2]; x.v[8] = q.x; x.v[9] = q.y; x.v[10] = q.z; x.v[11] = q.w;
    const uint32_t flags = x.v[11] >> 30;  // 2 = PositiveY, 1 = infinity
    x.v[11] &= 0x3fffffffu;
    bool ok = flags != 3 && fq_lt_mod(x);
    G1Affine p;
    p.x = fq_zero();
    p.y = fq_zero();
    if (flags & 1) {  // infinity: canonical only as x = 0 with the sign bit clear
      ok = ok && fq_is_zero(x);
    } else if (ok) {
      p.x = fq_to_mont(x);
      const Fq four = fq_dbl(fq_dbl(fq_one()));
      ok = fq_sqrt(fq_add(fq_mul(fq_sqr(p.x), p.x), four), &p.y);
      const Fq y = fq_from_mont(p.y);
      if (fq_gt_canon(y, fq_neg(y)) != ((flags & 2) != 0)) p.y = fq_neg(p.y);
      if (ok && check >= 2) ok = g1_in_subgroup(p);
    }
    fq_store(&out[i].x, p.x);
    fq_store(&out[i].y, p.y);
    if (ok_out) ok_out[i] = ok ? 1 : 0;
    if (!ok) {
      atomicAdd(bad, 1ull);
      atomicMin(bad + 1, (unsigned long long)i + 1);
    }
  }
}

// ---- Fr records (32 B little-endian canonical) ---------------------------------------------------------------------
// Montgomery scalars -> wire records, one scalar per thread as two 16-byte loads and stores.
__global__ void __launch_bounds__(128) k_fr_to_wire(const Fr* __restrict__ in, size_t len, Fr* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x)
    fr_store(out + i, fr_from_mont(fr_load(in + i)));
}

// Wire records -> Montgomery scalars; a record >= r is rejected (its slot gets zero).  bad[] as in k_g1_from_wire.
__global__ void __launch_bounds__(128) k_fr_from_wire(const Fr* __restrict__ in, size_t len, Fr* __restrict__ out,
                                                      unsigned long long* __restrict__ bad) {
  const uint32_t m[8] = TP_FR_MOD, r2c[8] = TP_FR_R2;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    const Fr a = fr_load(in + i);
    bool lt = false;
    for (int k = 7; k >= 0; k--) {
      if (a.v[k] != m[k]) {
        lt = a.v[k] < m[k];
        break;
      }
    }
    Fr r2;
#pragma unroll
    for (int k = 0; k < 8; k++) r2.v[k] = r2c[k];
    fr_store(out + i, lt ? fr_mul(a, r2) : fr_zero());
    if (!lt) {
      atomicAdd(bad, 1ull);
      atomicMin(bad + 1, (unsigned long long)i + 1);
    }
  }
}

static unsigned wire_grid(tp_ctx* ctx, size_t len) {
  size_t blocks = (len + 127) / 128;
  size_t cap = (size_t)ctx->sm_count * 16;
  return (unsigned)(blocks < cap ? (blocks ? blocks : 1) : cap);
}

int fr_to_wire_dev(tp_ctx* ctx, const Fr* in, size_t len, void* out_dev) {
  if (!len) return TP_OK;
  k_fr_to_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>(in, len, (Fr*)out_dev);
  TP_LAUNCH(ctx, "k_fr_to_wire");
  return TP_OK;
}

int fr_from_wire_dev(tp_ctx* ctx, const void* in_dev, size_t len, Fr* out, size_t* rejected, size_t* first_rejected) {
  *rejected = 0;
  *first_rejected = 0;
  if (!len) return TP_OK;
  TP_TRY(ensure(ctx, ctx->flag, 16));
  unsigned long long init[2] = {0, ~0ull}, got[2];
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->flag.p, init, 16, cudaMemcpyHostToDevice, ctx->stream));
  k_fr_from_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>((const Fr*)in_dev, len, out, (unsigned long long*)ctx->flag.p);
  TP_LAUNCH(ctx, "k_fr_from_wire");
  TP_CUDA_OK(ctx, cudaMemcpyAsync(got, ctx->flag.p, 16, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  *rejected = (size_t)got[0];
  *first_rejected = got[0] ? (size_t)(got[1] - 1) : 0;
  return TP_OK;
}

int g1_to_wire_dev(tp_ctx* ctx, const G1Affine* in, size_t len, void* out_dev) {
  if (!len) return TP_OK;
  k_g1_to_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>(in, len, (uint4*)out_dev);
  TP_LAUNCH(ctx, "k_g1_to_wire");
  return TP_OK;
}

int g1_from_wire_dev(tp_ctx* ctx, const void* in_dev, size_t len, int check, G1Affine* out, size_t* rejected,
                     size_t* first_rejected) {
  *rejected = 0;
  *first_rejected = 0;
  if (!len) return TP_OK;
  TP_TRY(ensure(ctx, ctx->flag, 16));
  unsigned long long init[2] = {0, ~0ull}, got[2];
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->flag.p, init, 16, cudaMemcpyHostToDevice, ctx->stream));
  k_g1_from_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>((const uint4*)in_dev, len, check, out,
                                                                (unsigned long long*)ctx->flag.p);
  TP_LAUNCH(ctx, "k_g1_from_wire");
  TP_CUDA_OK(ctx, cudaMemcpyAsync(got, ctx->flag.p, 16, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  *rejected = (size_t)got[0];
  *first_rejected = got[0] ? (size_t)(got[1] - 1) : 0;
  return TP_OK;
}

static int g1_to_wire_compressed_dev(tp_ctx* ctx, const G1Affine* in, size_t len, void* out_dev) {
  if (!len) return TP_OK;
  k_g1_to_wire_compressed<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>(in, len, (uint4*)out_dev);
  TP_LAUNCH(ctx, "k_g1_to_wire_compressed");
  return TP_OK;
}

// ok_dev (may be null): one byte per record, 1 = accepted.
static int g1_from_wire_compressed_dev(tp_ctx* ctx, const void* in_dev, size_t len, int check, G1Affine* out,
                                uint8_t* ok_dev, size_t* rejected, size_t* first_rejected) {
  *rejected = 0;
  *first_rejected = 0;
  if (!len) return TP_OK;
  TP_TRY(ensure(ctx, ctx->flag, 16));
  unsigned long long init[2] = {0, ~0ull}, got[2];
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->flag.p, init, 16, cudaMemcpyHostToDevice, ctx->stream));
  k_g1_from_wire_compressed<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>(
      (const uint4*)in_dev, len, check, out, (unsigned long long*)ctx->flag.p, ok_dev);
  TP_LAUNCH(ctx, "k_g1_from_wire_compressed");
  TP_CUDA_OK(ctx, cudaMemcpyAsync(got, ctx->flag.p, 16, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  *rejected = (size_t)got[0];
  *first_rejected = got[0] ? (size_t)(got[1] - 1) : 0;
  return TP_OK;
}

// ---- host side: single items ---------------------------------------------------------------------------------------
static void fq_to_wire(const HFq& a, uint8_t out[48]) {
  HFq c = a.from_mont();
  memcpy(out, c.v, 48);
}
static bool fq_from_wire(const uint8_t in[48], uint8_t flag_mask, HFq* out, uint8_t* flags) {
  uint64_t v[6];
  memcpy(v, in, 48);
  if (flags) *flags = (uint8_t)(v[5] >> 56) & flag_mask;
  v[5] &= ~((uint64_t)flag_mask << 56);
  if (ge<6>(v, FQ_PARAMS.mod)) return false;
  *out = HFq::to_mont(v);
  return true;
}

void g2_to_wire(const G2Aff& p, uint8_t out[TP_WIRE_G2_BYTES]) {
  if (p.inf) {
    memset(out, 0, TP_WIRE_G2_BYTES);
    out[96] = 1;
    out[191] |= 0x40;
    return;
  }
  fq_to_wire(p.x.a, out);
  fq_to_wire(p.x.b, out + 48);
  fq_to_wire(p.y.a, out + 96);
  fq_to_wire(p.y.b, out + 144);
}
bool g2_from_wire(const uint8_t in[TP_WIRE_G2_BYTES], int check, G2Aff* out) {
  uint8_t flags = 0;
  G2Aff p;
  p.inf = false;
  bool ok = fq_from_wire(in, 0, &p.x.a, nullptr) && fq_from_wire(in + 48, 0, &p.x.b, nullptr) &&
            fq_from_wire(in + 96, 0, &p.y.a, nullptr) && fq_from_wire(in + 144, 0xc0, &p.y.b, &flags);
  if (!ok || (flags & 0x80)) return false;
  if (flags & 0x40) {  // infinity is canonical only as (x, y) = (0, 1)
    if (!(p.x == Fq2::zero()) || !(p.y == Fq2::one())) return false;
    *out = {Fq2::zero(), Fq2::one(), true};
    return true;
  }
  if (check >= 1 && !g2_on_curve(p)) return false;
  if (check >= 2 && !g2_mul(p, FR_PARAMS.mod, 4).inf) return false;
  *out = p;
  return true;
}

static bool g1_wire_valid(const uint8_t in[TP_WIRE_G1_BYTES]) {
  uint8_t flags = 0;
  G1Aff p;
  p.inf = false;
  if (!fq_from_wire(in, 0, &p.x, nullptr) || !fq_from_wire(in + 48, 0xc0, &p.y, &flags)) return false;
  if (flags & 0x80) return false;
  if (flags & 0x40) return p.x == HFq::zero() && p.y == HFq::one();  // infinity is canonical only as (0, 1)
  return g1aff_on_curve(p);
}

// ---- host side: compressed items -----------------------------------------------------------------------------------
// sqrt(a) = a^((q+1)/4) (q = 3 mod 4); false if a is not a square.  Montgomery in and out.
static bool hfq_sqrt(const HFq& a, HFq* y) {
  uint64_t e[6], one[6] = {1, 0, 0, 0, 0, 0};
  add_n<6>(e, FQ_PARAMS.mod, one);
  for (int i = 0; i < 6; i++) e[i] = (e[i] >> 2) | (i < 5 ? e[i + 1] << 62 : 0);
  *y = a.pow(e, 6);
  return y->sqr() == a;
}
// y > -y comparing canonical integers (ark-ff's Ord on Fp)
static bool hfq_is_positive(const HFq& y) {
  HFq c = y.from_mont(), n = y.neg().from_mont();
  for (int i = 5; i >= 0; i--)
    if (c.v[i] != n.v[i]) return c.v[i] > n.v[i];
  return false;
}
// Fq2's order compares c1 first, then c0.  ⚠ Recalled from ark-ff 0.3 (QuadExtField's Ord), not checked offline.
static bool fq2_is_positive(const Fq2& y) {
  if (y.b != y.b.neg()) return hfq_is_positive(y.b);
  return hfq_is_positive(y.a);
}
static Fq2 fq2_pow(const Fq2& a, const uint64_t* e, int n) {
  Fq2 r = Fq2::one();
  for (int i = n - 1; i >= 0; i--)
    for (int b = 63; b >= 0; b--) {
      r = r.sqr();
      if ((e[i] >> b) & 1) r = r * a;
    }
  return r;
}
// Square root in Fq2 for q = 3 mod 4 (Adj and Rodriguez-Henriquez, "Square root computation over even extension
// fields", Algorithm 9); the result is checked by squaring, so a non-square is always reported.
static bool fq2_sqrt(const Fq2& a, Fq2* out) {
  if (a.is_zero()) {
    *out = Fq2::zero();
    return true;
  }
  uint64_t e1[6], e2[6], three[6] = {3, 0, 0, 0, 0, 0}, one[6] = {1, 0, 0, 0, 0, 0};
  sub_n<6>(e1, FQ_PARAMS.mod, three);  // (q - 3) / 4
  for (int i = 0; i < 6; i++) e1[i] = (e1[i] >> 2) | (i < 5 ? e1[i + 1] << 62 : 0);
  sub_n<6>(e2, FQ_PARAMS.mod, one);    // (q - 1) / 2
  for (int i = 0; i < 6; i++) e2[i] = (e2[i] >> 1) | (i < 5 ? e2[i + 1] << 63 : 0);
  const Fq2 a1 = fq2_pow(a, e1, 6);
  const Fq2 alpha = a1 * a1 * a;
  const Fq2 x0 = a1 * a;
  const Fq2 minus_one = Fq2::one().neg();
  Fq2 x;
  if (alpha == minus_one) {
    x = {x0.b.neg(), x0.a};  // u * x0
  } else {
    x = fq2_pow(Fq2::one() + alpha, e2, 6) * x0;
  }
  if (x.sqr() != a) return false;
  *out = x;
  return true;
}

// 96-byte uncompressed record (already validated) -> 48-byte compressed record
static void g1_wire_compress(const uint8_t in[TP_WIRE_G1_BYTES], uint8_t out[TP_WIRE_G1_COMPRESSED_BYTES]) {
  if (in[95] & 0x40) {
    memset(out, 0, TP_WIRE_G1_COMPRESSED_BYTES);
    out[47] = 0x40;
    return;
  }
  HFq y;
  fq_from_wire(in + 48, 0xc0, &y, nullptr);
  memcpy(out, in, TP_WIRE_G1_COMPRESSED_BYTES);
  if (hfq_is_positive(y)) out[47] |= 0x80;
}
// 48-byte compressed record -> 96-byte uncompressed record; false for x >= q, bad flags or an x without a root.
static bool g1_wire_decompress(const uint8_t in[TP_WIRE_G1_COMPRESSED_BYTES], uint8_t out[TP_WIRE_G1_BYTES]) {
  uint8_t flags = 0;
  HFq x;
  if (!fq_from_wire(in, 0xc0, &x, &flags) || flags == 0xc0) return false;
  if (flags & 0x40) {  // infinity: canonical only as x = 0 with the sign bit clear
    if (!x.is_zero()) return false;
    memset(out, 0, TP_WIRE_G1_BYTES);
    out[48] = 1;
    out[95] = 0x40;
    return true;
  }
  HFq y;
  if (!hfq_sqrt(x.sqr() * x + HFq::from_u64(4), &y)) return false;
  if (hfq_is_positive(y) != ((flags & 0x80) != 0)) y = y.neg();
  fq_to_wire(x, out);
  fq_to_wire(y, out + 48);
  return true;
}

static void g2_to_wire_compressed(const G2Aff& p, uint8_t out[TP_WIRE_G2_COMPRESSED_BYTES]) {
  if (p.inf) {
    memset(out, 0, TP_WIRE_G2_COMPRESSED_BYTES);
    out[95] = 0x40;
    return;
  }
  fq_to_wire(p.x.a, out);
  fq_to_wire(p.x.b, out + 48);
  if (fq2_is_positive(p.y)) out[95] |= 0x80;
}
static bool g2_from_wire_compressed(const uint8_t in[TP_WIRE_G2_COMPRESSED_BYTES], int check, G2Aff* out) {
  uint8_t flags = 0;
  G2Aff p;
  p.inf = false;
  if (!fq_from_wire(in, 0, &p.x.a, nullptr) || !fq_from_wire(in + 48, 0xc0, &p.x.b, &flags) || flags == 0xc0)
    return false;
  if (flags & 0x40) {
    if (!p.x.is_zero()) return false;
    *out = {Fq2::zero(), Fq2::one(), true};
    return true;
  }
  const Fq2 b = {HFq::from_u64(4), HFq::from_u64(4)};
  if (!fq2_sqrt(p.x.sqr() * p.x + b, &p.y)) return false;
  if (fq2_is_positive(p.y) != ((flags & 0x80) != 0)) p.y = p.y.neg();
  if (check >= 2 && !g2_mul(p, FR_PARAMS.mod, 4).inf) return false;
  *out = p;
  return true;
}

}  // namespace tp

// ---- the proof -----------------------------------------------------------------------------------------------------
// proof.rs:85-95 in the order tp_prove writes it: G = a G1 point, F = a scalar.
static const char kProofLayout[] = "GGF" "GGF" "GGF" "GGF" "GF" "F" "GGG" "GF";

extern "C" {

int tp_proof_encoded_size(size_t n_public, size_t* bytes) {
  if (!bytes) return TP_ERR_INVALID_ARG;
  *bytes = TP_PROOF_FIXED_BYTES + 8 + 32 * n_public;
  return TP_OK;
}

int tp_proof_encode(const uint8_t* fixed, const uint64_t* public_inputs, size_t n_public, uint8_t* out, size_t cap,
                    size_t* written) {
  if (!fixed || !out || (n_public && !public_inputs)) return TP_ERR_INVALID_ARG;
  const size_t need = TP_PROOF_FIXED_BYTES + 8 + 32 * n_public;
  if (written) *written = need;
  if (cap < need) return TP_ERR_BUFFER_TOO_SMALL;
  memcpy(out, fixed, TP_PROOF_FIXED_BYTES);
  uint64_t n64 = n_public;
  memcpy(out + TP_PROOF_FIXED_BYTES, &n64, 8);
  uint8_t* o = out + TP_PROOF_FIXED_BYTES + 8;
  for (size_t i = 0; i < n_public; i++, o += 32) {
    HFr v;
    memcpy(v.v, public_inputs + 4 * i, 32);
    if (ge<4>(v.v, FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
    HFr c = v.from_mont();
    memcpy(o, c.v, 32);
  }
  return TP_OK;
}

// ark-serialize's CHECKED deserialisation also verifies [r]P = 0 for every point; tp_proof_decode stops at "on the
// curve" (the reference's transcript uses the unchecked form).  This is the additional check, on the host: 13 scalar
// multiplications by r.
int tp_proof_points_in_subgroup(const uint8_t* fixed, size_t len, int* ok) {
  if (!fixed || !ok || len < TP_PROOF_FIXED_BYTES) return TP_ERR_INVALID_ARG;
  *ok = 0;
  const uint8_t* p = fixed;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k != 'G') {
      p += 32;
      continue;
    }
    if (!tp::g1_wire_valid(p)) return TP_ERR_MALFORMED;
    uint8_t flags = 0;
    G1Aff a;
    a.inf = false;
    tp::fq_from_wire(p, 0, &a.x, nullptr);
    tp::fq_from_wire(p + 48, 0xc0, &a.y, &flags);
    if (!(flags & 0x40)) {
      HG1 m = g1_mul_u64limbs(g1_from_affine(a.x, a.y), FR_PARAMS.mod, 4);
      if (!m.is_identity()) return TP_OK;   // *ok stays 0
    }
    p += TP_WIRE_G1_BYTES;
  }
  *ok = 1;
  return TP_OK;
}

int tp_proof_decode(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_FIXED_BYTES],
                    uint64_t* public_inputs_out, size_t cap_public, size_t* n_public) {
  if (!bytes || !n_public) return TP_ERR_INVALID_ARG;
  if (len < TP_PROOF_FIXED_BYTES + 8) return TP_ERR_MALFORMED;
  uint64_t n64;
  memcpy(&n64, bytes + TP_PROOF_FIXED_BYTES, 8);
  if (n64 > (len - TP_PROOF_FIXED_BYTES - 8) / 32 || len != TP_PROOF_FIXED_BYTES + 8 + 32 * (size_t)n64)
    return TP_ERR_MALFORMED;
  const uint8_t* p = bytes;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k == 'G') {
      if (!tp::g1_wire_valid(p)) return TP_ERR_MALFORMED;
      p += TP_WIRE_G1_BYTES;
    } else {
      uint64_t v[4];
      memcpy(v, p, 32);
      if (ge<4>(v, FR_PARAMS.mod)) return TP_ERR_MALFORMED;
      p += 32;
    }
  }
  p += 8;
  for (size_t i = 0; i < n64; i++) {
    uint64_t v[4];
    memcpy(v, p + 32 * i, 32);
    if (ge<4>(v, FR_PARAMS.mod)) return TP_ERR_MALFORMED;
  }
  *n_public = (size_t)n64;
  if (public_inputs_out) {
    if (cap_public < n64) return TP_ERR_BUFFER_TOO_SMALL;
    for (size_t i = 0; i < n64; i++) {
      uint64_t v[4];
      memcpy(v, p + 32 * i, 32);
      HFr m = HFr::to_mont(v);
      memcpy(public_inputs_out + 4 * i, m.v, 32);
    }
  }
  if (fixed_out) memcpy(fixed_out, bytes, TP_PROOF_FIXED_BYTES);
  return TP_OK;
}

// ---- the proof with compressed points: the same fields in the same order, 48 B per G1 point --------------------------
static bool fr_wire_valid(const uint8_t* p) {
  uint64_t v[4];
  memcpy(v, p, 32);
  return !ge<4>(v, FR_PARAMS.mod);
}

int tp_proof_compress(const uint8_t* fixed, size_t len, uint8_t* out, size_t cap) {
  if (!fixed || !out) return TP_ERR_INVALID_ARG;
  if (len != TP_PROOF_FIXED_BYTES) return TP_ERR_MALFORMED;
  if (cap < TP_PROOF_COMPRESSED_FIXED_BYTES) return TP_ERR_BUFFER_TOO_SMALL;
  const uint8_t* p = fixed;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k == 'G') {
      if (!tp::g1_wire_valid(p)) return TP_ERR_MALFORMED;
      p += TP_WIRE_G1_BYTES;
    } else {
      if (!fr_wire_valid(p)) return TP_ERR_MALFORMED;
      p += 32;
    }
  }
  p = fixed;
  uint8_t* o = out;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k == 'G') {
      tp::g1_wire_compress(p, o);
      p += TP_WIRE_G1_BYTES;
      o += TP_WIRE_G1_COMPRESSED_BYTES;
    } else {
      memcpy(o, p, 32);
      p += 32;
      o += 32;
    }
  }
  return TP_OK;
}

int tp_proof_decompress(const uint8_t* in, size_t len, uint8_t* fixed_out, size_t cap) {
  if (!in || !fixed_out) return TP_ERR_INVALID_ARG;
  if (len != TP_PROOF_COMPRESSED_FIXED_BYTES) return TP_ERR_MALFORMED;
  if (cap < TP_PROOF_FIXED_BYTES) return TP_ERR_BUFFER_TOO_SMALL;
  uint8_t tmp[TP_PROOF_FIXED_BYTES];
  const uint8_t* p = in;
  uint8_t* o = tmp;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k == 'G') {
      if (!tp::g1_wire_decompress(p, o)) return TP_ERR_MALFORMED;
      p += TP_WIRE_G1_COMPRESSED_BYTES;
      o += TP_WIRE_G1_BYTES;
    } else {
      if (!fr_wire_valid(p)) return TP_ERR_MALFORMED;
      memcpy(o, p, 32);
      p += 32;
      o += 32;
    }
  }
  memcpy(fixed_out, tmp, TP_PROOF_FIXED_BYTES);
  return TP_OK;
}

int tp_proof_encoded_size_compressed(size_t n_public, size_t* bytes) {
  if (!bytes) return TP_ERR_INVALID_ARG;
  *bytes = TP_PROOF_COMPRESSED_FIXED_BYTES + 8 + 32 * n_public;
  return TP_OK;
}

int tp_proof_encode_compressed(const uint8_t* fixed, const uint64_t* public_inputs, size_t n_public, uint8_t* out,
                               size_t cap, size_t* written) {
  if (!fixed || !out || (n_public && !public_inputs)) return TP_ERR_INVALID_ARG;
  const size_t need = TP_PROOF_COMPRESSED_FIXED_BYTES + 8 + 32 * n_public;
  if (written) *written = need;
  if (cap < need) return TP_ERR_BUFFER_TOO_SMALL;
  // the tail is the uncompressed encoder's: encode the Vec<Fr> behind a scratch block, then move it
  std::vector<uint8_t> full(TP_PROOF_FIXED_BYTES + 8 + 32 * n_public);
  TP_TRY(tp_proof_encode(fixed, public_inputs, n_public, full.data(), full.size(), nullptr));
  TP_TRY(tp_proof_compress(fixed, TP_PROOF_FIXED_BYTES, out, cap));
  memcpy(out + TP_PROOF_COMPRESSED_FIXED_BYTES, full.data() + TP_PROOF_FIXED_BYTES, 8 + 32 * n_public);
  return TP_OK;
}

int tp_proof_decode_compressed(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_FIXED_BYTES],
                               uint64_t* public_inputs_out, size_t cap_public, size_t* n_public) {
  if (!bytes || !n_public) return TP_ERR_INVALID_ARG;
  if (len < TP_PROOF_COMPRESSED_FIXED_BYTES + 8) return TP_ERR_MALFORMED;
  uint64_t n64;
  memcpy(&n64, bytes + TP_PROOF_COMPRESSED_FIXED_BYTES, 8);
  if (n64 > (len - TP_PROOF_COMPRESSED_FIXED_BYTES - 8) / 32 ||
      len != TP_PROOF_COMPRESSED_FIXED_BYTES + 8 + 32 * (size_t)n64)
    return TP_ERR_MALFORMED;
  // the uncompressed decoder checks the Vec<Fr> and converts it: decode the equivalent uncompressed encoding
  std::vector<uint8_t> full(TP_PROOF_FIXED_BYTES + 8 + 32 * (size_t)n64);
  TP_TRY(tp_proof_decompress(bytes, TP_PROOF_COMPRESSED_FIXED_BYTES, full.data(), TP_PROOF_FIXED_BYTES));
  memcpy(full.data() + TP_PROOF_FIXED_BYTES, bytes + TP_PROOF_COMPRESSED_FIXED_BYTES, 8 + 32 * (size_t)n64);
  return tp_proof_decode(full.data(), full.size(), fixed_out, public_inputs_out, cap_public, n_public);
}

// Many compressed blocks at once: the 13 x-records of every block go through the device (one square root per thread),
// the recovered points come back uncompressed; the host checks the scalars and assembles the blocks.
int tp_proofs_decompress(tp_ctx* ctx, const uint8_t* in, size_t count, uint8_t* fixed_out, size_t cap, int* status) {
  if (!ctx || count > 65536 || (count && (!in || !fixed_out))) return TP_ERR_INVALID_ARG;
  if (!count) return TP_OK;
  if (cap < count * TP_PROOF_FIXED_BYTES) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "proofs_decompress: output buffer too small");
  if (!ctx->children.empty())   // device group: rank 0 does the work
    return group_run(ctx, [&](tp_ctx* c, int r) { return r == 0 ? tp_proofs_decompress(c, in, count, fixed_out, cap, status) : TP_OK; });
  const size_t kPoints = 13;
  const size_t npts = count * kPoints;
  std::vector<uint8_t> xs(npts * TP_WIRE_G1_COMPRESSED_BYTES), pts(npts * TP_WIRE_G1_BYTES), oks(npts);
  for (size_t k = 0; k < count; k++) {
    const uint8_t* p = in + k * TP_PROOF_COMPRESSED_FIXED_BYTES;
    uint8_t* x = xs.data() + k * kPoints * TP_WIRE_G1_COMPRESSED_BYTES;
    for (const char* f = kProofLayout; *f; f++) {
      if (*f == 'G') {
        memcpy(x, p, TP_WIRE_G1_COMPRESSED_BYTES);
        x += TP_WIRE_G1_COMPRESSED_BYTES;
        p += TP_WIRE_G1_COMPRESSED_BYTES;
      } else {
        p += 32;
      }
    }
  }
  // one allocation: x-records | Montgomery points | uncompressed records | ok bytes
  const size_t off_aff = (npts * TP_WIRE_G1_COMPRESSED_BYTES + 255) & ~(size_t)255;
  const size_t off_wire = off_aff + npts * sizeof(G1Affine);
  const size_t off_ok = off_wire + npts * TP_WIRE_G1_BYTES;
  void* stage = nullptr;
  if (cudaMalloc(&stage, off_ok + npts) != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, TP_ERR_CUDA, "proofs_decompress: out of device memory");
  }
  uint8_t* base = (uint8_t*)stage;
  size_t rejected = 0, first = 0;
  int rc = TP_OK;
  if (cudaMemcpyAsync(base, xs.data(), xs.size(), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
    rc = fail(ctx, TP_ERR_CUDA, "proofs_decompress: copy failed");
  if (rc == TP_OK)
    rc = g1_from_wire_compressed_dev(ctx, base, npts, 1, (G1Affine*)(base + off_aff), base + off_ok, &rejected, &first);
  if (rc == TP_OK) rc = g1_to_wire_dev(ctx, (const G1Affine*)(base + off_aff), npts, base + off_wire);
  if (rc == TP_OK &&
      (cudaMemcpyAsync(pts.data(), base + off_wire, pts.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
       cudaMemcpyAsync(oks.data(), base + off_ok, npts, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
       cudaStreamSynchronize(ctx->stream) != cudaSuccess))
    rc = fail(ctx, TP_ERR_CUDA, "proofs_decompress: copy failed");
  cudaFree(stage);
  if (rc != TP_OK) return rc;
  size_t first_bad = count;
  for (size_t k = 0; k < count; k++) {
    const uint8_t* p = in + k * TP_PROOF_COMPRESSED_FIXED_BYTES;
    const uint8_t* pt = pts.data() + k * kPoints * TP_WIRE_G1_BYTES;
    const uint8_t* ok = oks.data() + k * kPoints;
    uint8_t* o = fixed_out + k * TP_PROOF_FIXED_BYTES;
    bool good = true;
    for (const char* f = kProofLayout; *f; f++) {
      if (*f == 'G') {
        good = good && *ok++;
        memcpy(o, pt, TP_WIRE_G1_BYTES);
        pt += TP_WIRE_G1_BYTES;
        o += TP_WIRE_G1_BYTES;
        p += TP_WIRE_G1_COMPRESSED_BYTES;
      } else {
        good = good && fr_wire_valid(p);
        memcpy(o, p, 32);
        o += 32;
        p += 32;
      }
    }
    if (!good) {
      memset(fixed_out + k * TP_PROOF_FIXED_BYTES, 0, TP_PROOF_FIXED_BYTES);
      if (first_bad == count) first_bad = k;
    }
    if (status) status[k] = good ? TP_OK : TP_ERR_MALFORMED;
  }
  if (!status && first_bad < count) {
    ctx->err = "proofs_decompress: proof " + std::to_string(first_bad) + " is malformed";
    return TP_ERR_MALFORMED;
  }
  return TP_OK;
}

}  // extern "C"

// ---- the SRS -------------------------------------------------------------------------------------------------------
// Srs = u64 count | count G1 records | G2 | tau G2, in either encoding: only the record sizes, the device conversion of
// the G1 records and the host G2 codec depend on it.
namespace {

struct SrsEncoding {
  bool compressed;
  const char* ser;   // names in tp_last_error
  const char* de;
  size_t g1_bytes() const { return compressed ? TP_WIRE_G1_COMPRESSED_BYTES : TP_WIRE_G1_BYTES; }
  size_t g2_bytes() const { return compressed ? TP_WIRE_G2_COMPRESSED_BYTES : TP_WIRE_G2_BYTES; }
  size_t size(size_t len) const { return 8 + len * g1_bytes() + 2 * g2_bytes(); }
};
const SrsEncoding kUncompressed = {false, "srs_serialize", "srs_deserialize"};
const SrsEncoding kCompressed = {true, "srs_serialize_compressed", "srs_deserialize_compressed"};

int srs_fail(tp_ctx* ctx, int code, const char* fn, const char* msg) {
  ctx->err = std::string(fn) + ": " + msg;
  return code;
}

int srs_serialize_as(const SrsEncoding& enc, tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written) {
  if (!ctx || !srs || !out) return TP_ERR_INVALID_ARG;
  if (!ctx->children.empty())   // device group: rank 0's copy
    return group_run(ctx, [&](tp_ctx* c, int r) { return r == 0 ? srs_serialize_as(enc, c, srs->parts[0], out, cap, written) : TP_OK; });
  if (!srs->pairing) return srs_fail(ctx, TP_ERR_INVALID_ARG, enc.ser, "the SRS has no G2 points (tp_srs_set_g2)");
  const size_t need = enc.size(srs->len);
  if (written) *written = need;
  if (cap < need) return srs_fail(ctx, TP_ERR_BUFFER_TOO_SMALL, enc.ser, "output buffer too small");
  uint64_t n64 = srs->len;
  memcpy(out, &n64, 8);
  if (srs->len) {
    void* stage = nullptr;
    TP_CUDA_OK(ctx, cudaMalloc(&stage, srs->len * enc.g1_bytes()));
    int rc = enc.compressed ? g1_to_wire_compressed_dev(ctx, srs->g1, srs->len, stage) : g1_to_wire_dev(ctx, srs->g1, srs->len, stage);
    if (rc == TP_OK && (cudaMemcpyAsync(out + 8, stage, srs->len * enc.g1_bytes(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                        cudaStreamSynchronize(ctx->stream) != cudaSuccess))
      rc = srs_fail(ctx, TP_ERR_CUDA, enc.ser, "copy failed");
    cudaFree(stage);
    if (rc != TP_OK) return rc;
  }
  uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
  if (tp_srs_g2(srs, g2, g2s) != TP_OK) return srs_fail(ctx, TP_ERR_INVALID_ARG, enc.ser, "no G2 points");
  uint8_t* o = out + 8 + srs->len * enc.g1_bytes();
  if (enc.compressed) {
    g2_to_wire_compressed(g2_decode(g2), o);
    g2_to_wire_compressed(g2_decode(g2s), o + enc.g2_bytes());
  } else {
    g2_to_wire(g2_decode(g2), o);
    g2_to_wire(g2_decode(g2s), o + enc.g2_bytes());
  }
  return TP_OK;
}

int srs_deserialize_as(const SrsEncoding& enc, tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out) {
  if (!ctx || !bytes || !out || check < 0 || check > 2) return TP_ERR_INVALID_ARG;
  if (!ctx->children.empty()) {   // device group: every rank decodes (and validates) its own copy
    tp_srs* front = new tp_srs();
    front->parts.assign(ctx->children.size(), nullptr);
    int rc = group_run(ctx, [&](tp_ctx* c, int r) { return srs_deserialize_as(enc, c, bytes, len, check, &front->parts[r]); });
    if (rc != TP_OK) {
      group_run(ctx, [&](tp_ctx* c, int r) { return tp_srs_destroy(c, front->parts[r]); });
      delete front;
      return rc;
    }
    front->len = front->parts[0]->len;
    *out = front;
    return TP_OK;
  }
  if (len < enc.size(0)) return srs_fail(ctx, TP_ERR_MALFORMED, enc.de, "truncated");
  uint64_t n64;
  memcpy(&n64, bytes, 8);
  const size_t body = len - enc.size(0);
  if (n64 > body / enc.g1_bytes() || body != (size_t)n64 * enc.g1_bytes())
    return srs_fail(ctx, TP_ERR_MALFORMED, enc.de, "length does not match the point count");
  const size_t n = (size_t)n64;
  G2Aff q, qs;
  const uint8_t* tail = bytes + 8 + n * enc.g1_bytes();
  const bool g2_ok = enc.compressed ? g2_from_wire_compressed(tail, check, &q) && g2_from_wire_compressed(tail + enc.g2_bytes(), check, &qs)
                                    : g2_from_wire(tail, check, &q) && g2_from_wire(tail + enc.g2_bytes(), check, &qs);
  if (!g2_ok) return srs_fail(ctx, TP_ERR_MALFORMED, enc.de, "bad G2 point");
  tp_srs* s = nullptr;
  TP_TRY(srs_alloc(ctx, n, &s));
  int rc = TP_OK;
  size_t rejected = 0, first = 0;
  if (n) {
    void* stage = nullptr;
    if (cudaMalloc(&stage, n * enc.g1_bytes()) != cudaSuccess) {
      cudaGetLastError();
      rc = srs_fail(ctx, TP_ERR_CUDA, enc.de, "out of device memory");
    }
    if (rc == TP_OK && cudaMemcpyAsync(stage, bytes + 8, n * enc.g1_bytes(), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
      rc = srs_fail(ctx, TP_ERR_CUDA, enc.de, "copy failed");
    if (rc == TP_OK)
      rc = enc.compressed ? g1_from_wire_compressed_dev(ctx, stage, n, check, s->g1, nullptr, &rejected, &first)
                          : g1_from_wire_dev(ctx, stage, n, check, s->g1, &rejected, &first);
    if (stage) cudaFree(stage);
    if (rc == TP_OK && rejected) {
      ctx->err = std::string(enc.de) + ": " + std::to_string(rejected) + " G1 point(s) rejected, first at index " +
                 std::to_string(first);
      rc = TP_ERR_MALFORMED;
    }
  }
  if (rc == TP_OK) rc = srs_build_levels_dev(ctx, s);
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = srs_fail(ctx, TP_ERR_CUDA, enc.de, "failed");
  if (rc == TP_OK) {
    uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
    g2_encode(q, g2);
    g2_encode(qs, g2s);
    if (tp_srs_set_g2(s, g2, g2s) != TP_OK) rc = srs_fail(ctx, TP_ERR_MALFORMED, enc.de, "G2 points rejected");
  }
  if (rc != TP_OK) {
    tp_srs_destroy(ctx, s);
    return rc;
  }
  *out = s;
  return TP_OK;
}

}  // namespace

extern "C" {

int tp_srs_serialized_size(const tp_srs* srs, size_t* bytes) {
  if (!srs || !bytes) return TP_ERR_INVALID_ARG;
  *bytes = kUncompressed.size(srs->len);
  return TP_OK;
}
int tp_srs_serialize(tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written) {
  return srs_serialize_as(kUncompressed, ctx, srs, out, cap, written);
}
int tp_srs_deserialize(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out) {
  return srs_deserialize_as(kUncompressed, ctx, bytes, len, check, out);
}

// compressed points: u64 count | count x 48 B | G2 | tau G2 (96 B each)
int tp_srs_serialized_size_compressed(const tp_srs* srs, size_t* bytes) {
  if (!srs || !bytes) return TP_ERR_INVALID_ARG;
  *bytes = kCompressed.size(srs->len);
  return TP_OK;
}
int tp_srs_serialize_compressed(tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written) {
  return srs_serialize_as(kCompressed, ctx, srs, out, cap, written);
}
int tp_srs_deserialize_compressed(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out) {
  return srs_deserialize_as(kCompressed, ctx, bytes, len, check, out);
}

}  // extern "C"
