// BLS12-381 Fr / Fq device arithmetic for sm_100a: Montgomery form on 32-bit limbs
// (R = 2^256 / 2^384, little-endian), bit-compatible with ark_ff::Fp256 / Fp384 as the
// reference holds them in memory (SURVEY.md 8(b)); replaces the un-vendored ark-ff 0.3.0
// field types used throughout kzg/src/lib.rs, permutation/src/proving.rs and
// plonk/src/proof.rs.  The multiply/add/sub carry chains are generated inline PTX
// (mont_gen.cuh, tools/gen_mont.py).
#pragma once
#include <stdint.h>
#include "mont_gen.cuh"

namespace tp {

struct alignas(16) Fr {
  uint32_t v[8];
};
struct alignas(16) Fq {
  uint32_t v[12];
};

// ---- constants (Montgomery form) ----------------------------------------------------
// TP_FR_ONE / TP_FQ_ONE / TP_*_MOD / TP_*_MODM2 come from mont_gen.cuh (generated).

// ---- Fr -----------------------------------------------------------------------------
__device__ __forceinline__ Fr fr_zero() {
  Fr r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = 0;
  return r;
}
__device__ __forceinline__ Fr fr_one() {
  const uint32_t c[8] = TP_FR_ONE;
  Fr r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = c[i];
  return r;
}
__device__ __forceinline__ Fr fr_mul(const Fr& a, const Fr& b) {
  Fr r;
  fr_mul_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fr fr_sqr(const Fr& a) { return fr_mul(a, a); }
__device__ __forceinline__ Fr fr_add(const Fr& a, const Fr& b) {
  Fr r;
  fr_add_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fr fr_sub(const Fr& a, const Fr& b) {
  Fr r;
  fr_sub_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fr fr_neg(const Fr& a) { return fr_sub(fr_zero(), a); }
// Lazy forms (values in [0, 2r), 2r < 2^256; tools/gen_mont.py build_add2): the product keeps its result unreduced --
// `w` must be the REDUCED operand (< r), `x` may be lazy -- sums and differences are taken modulo 2r, fr_norm2 returns
// to [0, r).  fr_mul(w, x) with a lazy x is also fine and returns a canonical value.
__device__ __forceinline__ Fr fr_mul_lazy(const Fr& w, const Fr& x) {
  Fr r;
  fr_mul_lazy_ptx(r.v, w.v, x.v);
  return r;
}
__device__ __forceinline__ Fr fr_add2(const Fr& a, const Fr& b) {
  Fr r;
  fr_add2_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fr fr_sub2(const Fr& a, const Fr& b) {
  Fr r;
  fr_sub2_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fr fr_norm2(const Fr& a) {
  Fr r;
  fr_norm2_ptx(r.v, a.v);
  return r;
}
__device__ __forceinline__ Fr fr_dbl(const Fr& a) { return fr_add(a, a); }
__device__ __forceinline__ bool fr_is_zero(const Fr& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i];
  return o == 0;
}
__device__ __forceinline__ bool fr_eq(const Fr& a, const Fr& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.v[i] ^ b.v[i];
  return o == 0;
}
// Montgomery -> canonical integer (multiply by 1).
__device__ __forceinline__ Fr fr_from_mont(const Fr& a) {
  Fr one_raw = fr_zero();
  one_raw.v[0] = 1;
  return fr_mul(a, one_raw);
}
// a^e for a 256-bit little-endian exponent held in e[8] (MSB-first square and multiply).
static __device__ __noinline__ Fr fr_pow(const Fr& a, const uint32_t* e, int nlimbs) {
  Fr r = fr_one();
  bool started = false;
  for (int i = nlimbs - 1; i >= 0; i--) {
    for (int b = 31; b >= 0; b--) {
      if (started) r = fr_sqr(r);
      if ((e[i] >> b) & 1) {
        r = started ? fr_mul(r, a) : a;
        started = true;
      }
    }
  }
  return r;
}
// Fermat inversion a^(r-2); returns 0 for 0 (callers check for zero where the reference panics).
static __device__ __noinline__ Fr fr_inv(const Fr& a) {
  const uint32_t e[8] = TP_FR_MODM2;
  return fr_pow(a, e, 8);
}
__device__ __forceinline__ Fr fr_pow_u64(const Fr& a, unsigned long long e) {
  uint32_t ee[2] = {(uint32_t)e, (uint32_t)(e >> 32)};
  return fr_pow(a, ee, 2);
}

__device__ __forceinline__ Fr fr_load(const Fr* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 lo = q[0], hi = q[1];
  Fr r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
__device__ __forceinline__ void fr_store(Fr* p, const Fr& a) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
}

// ---- Fq -----------------------------------------------------------------------------
__device__ __forceinline__ Fq fq_zero() {
  Fq r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = 0;
  return r;
}
__device__ __forceinline__ Fq fq_one() {
  const uint32_t c[12] = TP_FQ_ONE;
  Fq r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = c[i];
  return r;
}
// Multiplier forms (profiles/r1_summary.md, section J): TP_FQ_MUL_FORM 0 = interleaved CIOS
// (288 wide products), 1 = one-level Karatsuba wide product + separate reduction (252), 2 =
// schoolbook wide product + separate reduction (288; only for the microbenchmark).
#ifndef TP_FQ_MUL_FORM
#define TP_FQ_MUL_FORM 0
#endif
#ifdef TP_FQ_MUL_CALL
// One shared copy of the 381-bit product (keeps hot loops inside the instruction cache).
static __device__ __noinline__ Fq fq_mul(Fq a, Fq b) {
  Fq r;
  fq_mul_ptx(r.v, a.v, b.v);
  return r;
}
#else
__device__ __forceinline__ Fq fq_mul(const Fq& a, const Fq& b) {
  Fq r;
#if TP_FQ_MUL_FORM == 1
  fq_mul_kar_ptx(r.v, a.v, b.v);
#elif TP_FQ_MUL_FORM == 2
  fq_mul_sep_ptx(r.v, a.v, b.v);
#else
  fq_mul_ptx(r.v, a.v, b.v);
#endif
  return r;
}
#endif
// Dedicated square: 78 + 144 wide products instead of 288.
__device__ __forceinline__ Fq fq_sqr(const Fq& a) {
#ifdef TP_FQ_SQR_AS_MUL
  return fq_mul(a, a);
#else
  Fq r;
  fq_sqr_ptx(r.v, a.v);
  return r;
#endif
}
__device__ __forceinline__ Fq fq_add(const Fq& a, const Fq& b) {
  Fq r;
  fq_add_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fq fq_sub(const Fq& a, const Fq& b) {
  Fq r;
  fq_sub_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fq fq_neg(const Fq& a) { return fq_sub(fq_zero(), a); }
// a*b - c*d with ONE Montgomery reduction (lazy pair, 432 wide products instead of 576).  The
// subtrahend enters as c * (q - d); q - d lies in [1, q], which the pair's bound 2 q^2 < q 2^384 allows.
__device__ __forceinline__ Fq fq_mul_sub2(const Fq& a, const Fq& b, const Fq& c, const Fq& d) {
#ifdef TP_FQ_NO_LAZY
  return fq_sub(fq_mul(a, b), fq_mul(c, d));
#else
  const uint32_t q[12] = TP_FQ_MOD;
  Fq nd, r;
  asm("sub.cc.u32 %0, %12, %24;\n\t"
      "subc.cc.u32 %1, %13, %25;\n\t"
      "subc.cc.u32 %2, %14, %26;\n\t"
      "subc.cc.u32 %3, %15, %27;\n\t"
      "subc.cc.u32 %4, %16, %28;\n\t"
      "subc.cc.u32 %5, %17, %29;\n\t"
      "subc.cc.u32 %6, %18, %30;\n\t"
      "subc.cc.u32 %7, %19, %31;\n\t"
      "subc.cc.u32 %8, %20, %32;\n\t"
      "subc.cc.u32 %9, %21, %33;\n\t"
      "subc.cc.u32 %10, %22, %34;\n\t"
      "subc.u32 %11, %23, %35;"
      : "=r"(nd.v[0]), "=r"(nd.v[1]), "=r"(nd.v[2]), "=r"(nd.v[3]), "=r"(nd.v[4]), "=r"(nd.v[5]), "=r"(nd.v[6]),
        "=r"(nd.v[7]), "=r"(nd.v[8]), "=r"(nd.v[9]), "=r"(nd.v[10]), "=r"(nd.v[11])
      : "r"(q[0]), "r"(q[1]), "r"(q[2]), "r"(q[3]), "r"(q[4]), "r"(q[5]), "r"(q[6]), "r"(q[7]), "r"(q[8]), "r"(q[9]),
        "r"(q[10]), "r"(q[11]), "r"(d.v[0]), "r"(d.v[1]), "r"(d.v[2]), "r"(d.v[3]), "r"(d.v[4]), "r"(d.v[5]),
        "r"(d.v[6]), "r"(d.v[7]), "r"(d.v[8]), "r"(d.v[9]), "r"(d.v[10]), "r"(d.v[11]));
#if TP_FQ_MUL_FORM == 1
  fq_mul2_kar_ptx(r.v, a.v, b.v, c.v, nd.v);
#else
  fq_mul2_ptx(r.v, a.v, b.v, c.v, nd.v);
#endif
  return r;
#endif
}
__device__ __forceinline__ Fq fq_dbl(const Fq& a) { return fq_add(a, a); }
__device__ __forceinline__ bool fq_is_zero(const Fq& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) o |= a.v[i];
  return o == 0;
}
__device__ __forceinline__ bool fq_eq(const Fq& a, const Fq& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) o |= a.v[i] ^ b.v[i];
  return o == 0;
}
// Lazy forms for the MSM's addition laws (tools/gen_mont.py build_kq_minus): values in [0, 2q), 8q < 2^384.  Products
// of operands below 2q, and the pair a b - c d with c, d below 2q, come out below 2q without the final subtraction
// (either operand order: the simulator checks both); sums and differences are taken modulo 2q; fq_norm2 returns to
// [0, q).  Canonical values are valid lazy inputs.
__device__ __forceinline__ Fq fq_mul_lazy(const Fq& a, const Fq& b) {
  Fq r;
  fq_mul_lazy_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fq fq_sqr_lazy(const Fq& a) {
  Fq r;
  fq_sqr_lazy_ptx(r.v, a.v);
  return r;
}
// a b - c d = a b + c (2q - d): 2q - d lies in (0, 2q], 4 q^2 + 4 q^2 < q 2^384
__device__ __forceinline__ Fq fq_mul_sub2_lazy(const Fq& a, const Fq& b, const Fq& c, const Fq& d) {
  Fq nd, r;
  fq_neg2_ptx(nd.v, d.v);
  fq_mul2_lazy_ptx(r.v, a.v, b.v, c.v, nd.v);
  return r;
}
__device__ __forceinline__ Fq fq_add2(const Fq& a, const Fq& b) {
  Fq r;
  fq_add2_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fq fq_sub2(const Fq& a, const Fq& b) {
  Fq r;
  fq_sub2_ptx(r.v, a.v, b.v);
  return r;
}
__device__ __forceinline__ Fq fq_dbl2(const Fq& a) { return fq_add2(a, a); }
// q - a for a canonical a: in [1, q], no correction
__device__ __forceinline__ Fq fq_neg_lazy(const Fq& a) {
  Fq r;
  fq_neg1_ptx(r.v, a.v);
  return r;
}
__device__ __forceinline__ Fq fq_norm2(const Fq& a) {
  Fq r;
  fq_norm2_ptx(r.v, a.v);
  return r;
}
// a = 0 mod q for a in [0, 2q), i.e. a is 0 or q.  The low limb filters: the full compare runs only when it is the low
// limb of 0 or of q, which a non-zero value almost never has.
__device__ __forceinline__ bool fq_is_zero2(const Fq& a) {
  const uint32_t q[12] = TP_FQ_MOD;
  if (a.v[0] != 0 && a.v[0] != q[0]) return false;
  uint32_t oz = 0, oq = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    oz |= a.v[i];
    oq |= a.v[i] ^ q[i];
  }
  return oz == 0 || oq == 0;
}
static __device__ __noinline__ Fq fq_inv(const Fq& a) {
  const uint32_t e[12] = TP_FQ_MODM2;
  Fq r = fq_one();
  bool started = false;
  for (int i = 11; i >= 0; i--) {
    for (int b = 31; b >= 0; b--) {
      if (started) r = fq_sqr(r);
      if ((e[i] >> b) & 1) {
        r = started ? fq_mul(r, a) : a;
        started = true;
      }
    }
  }
  return r;
}
__device__ __forceinline__ Fq fq_load(const Fq* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1], c = q[2];
  Fq r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  r.v[8] = c.x; r.v[9] = c.y; r.v[10] = c.z; r.v[11] = c.w;
  return r;
}
__device__ __forceinline__ void fq_store(Fq* p, const Fq& a) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
  q[2] = make_uint4(a.v[8], a.v[9], a.v[10], a.v[11]);
}

}  // namespace tp
