// BLS12-381 G1 device arithmetic in XYZZ coordinates (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2;
// identity <=> ZZ == 0), a = 0, b = 4.  Replaces ark-ec 0.3.0 `GroupAffine::mul` /
// `GroupProjective` additions behind kzg/src/lib.rs:46-53 and kzg/src/srs.rs:15-24.
// Mixed addition = 8M + 2S, general addition = 12M + 2S, doubling = 6M + 3S (Fq).
#pragma once
#include "field.cuh"
#include "fq_inv.cuh"

namespace tp {

// Packed affine point as stored in the device SRS: (x, y) Montgomery, 96 bytes.
// (0, 0) encodes the point at infinity (it is not on y^2 = x^3 + 4).
struct alignas(16) G1Affine {
  Fq x, y;
};
struct alignas(16) G1Xyzz {
  Fq x, y, zz, zzz;
};

__device__ __forceinline__ G1Xyzz xyzz_identity() {
  G1Xyzz r;
  r.x = fq_zero(); r.y = fq_zero(); r.zz = fq_zero(); r.zzz = fq_zero();
  return r;
}
__device__ __forceinline__ bool xyzz_is_identity(const G1Xyzz& p) { return fq_is_zero(p.zz); }
__device__ __forceinline__ bool affine_is_identity(const G1Affine& p) { return fq_is_zero(p.x) && fq_is_zero(p.y); }

__device__ __forceinline__ G1Affine affine_load(const G1Affine* p) {
  G1Affine r;
  r.x = fq_load(&p->x);
  r.y = fq_load(&p->y);
  return r;
}
__device__ __forceinline__ void xyzz_store(G1Xyzz* p, const G1Xyzz& a) {
  fq_store(&p->x, a.x); fq_store(&p->y, a.y); fq_store(&p->zz, a.zz); fq_store(&p->zzz, a.zzz);
}
__device__ __forceinline__ G1Xyzz xyzz_load(const G1Xyzz* p) {
  G1Xyzz r;
  r.x = fq_load(&p->x); r.y = fq_load(&p->y); r.zz = fq_load(&p->zz); r.zzz = fq_load(&p->zzz);
  return r;
}

// Montgomery-form inverse by division steps (fq_inv.cuh); Fermat only if those did not terminate.
static __device__ __noinline__ Fq fq_inverse(const Fq& a) {
  Fq plain, r;
  if (!fqinv_plain(a.v, plain.v)) return fq_inv(a);
  const uint32_t r3[12] = FQINV_R3;
  Fq k;
#pragma unroll
  for (int i = 0; i < 12; i++) k.v[i] = r3[i];
  r = fq_mul(plain, k);   // (a R)^-1 * R^3 / R = a^-1 R
  return r;
}

// ---- affine pair addition with a shared (batched) inversion ------------------------------
// kind of a pair P1 + P2: 0 = chord (denominator x2 - x1), 1 = tangent (denominator 2 y1),
// 2 = result is the identity, 3 = result P1 (P2 is the identity), 4 = result P2.
// For kinds >= 2 the denominator is 1 so that it can sit in the running product.
static __device__ __noinline__ int affine_pair_special(const G1Affine& p1, const G1Affine& p2, Fq& d) {
  d = fq_one();
  if (affine_is_identity(p1)) return 4;
  if (affine_is_identity(p2)) return 3;
  if (fq_eq(p1.x, p2.x)) {
    if (fq_eq(p1.y, p2.y) && !fq_is_zero(p1.y)) {
      d = fq_dbl(p1.y);
      return 1;
    }
    return 2;
  }
  d = fq_sub(p2.x, p1.x);  // x = 0 on a non-identity point: an ordinary chord after all
  return 0;
}
// P1 + P2 given dinv = 1 / (denominator of `kind`); all cases of affine_pair_special.
__device__ __forceinline__ G1Affine affine_pair_finish(const G1Affine& p1, const G1Affine& p2, int kind, const Fq& dinv) {
  if (kind >= 2) {
    G1Affine r;
    if (kind == 3) return p1;
    if (kind == 4) return p2;
    r.x = fq_zero();
    r.y = fq_zero();
    return r;
  }
  Fq num;
  if (kind == 0) {
    num = fq_sub(p2.y, p1.y);
  } else {
    Fq xx = fq_sqr(p1.x);
    num = fq_add(fq_dbl(xx), xx);
  }
  Fq lam = fq_mul(num, dinv);
  G1Affine r;
  r.x = fq_sub(fq_sub(fq_sqr(lam), p1.x), p2.x);
  r.y = fq_sub(fq_mul(lam, fq_sub(p1.x, r.x)), p1.y);
  return r;
}

// Field arithmetic of the XYZZ laws.  Canonical (LAZY = false): every value in [0, q), as SRS generation, wire checks
// and the verifier use them.  Lazy (the MSM, msm.cu): every value in [0, 2q) -- products without their final
// subtraction, sums and differences modulo 2q (field.cuh) -- and stored so; the MSM brings its outputs to [0, q) with
// fq_norm2 before they leave the device.  The bounds in the comments of the laws are those of the lazy form.
template <bool LAZY> struct FqOps;
template <> struct FqOps<false> {
  static __device__ __forceinline__ Fq mul(const Fq& a, const Fq& b) { return fq_mul(a, b); }
  static __device__ __forceinline__ Fq sqr(const Fq& a) { return fq_sqr(a); }
  static __device__ __forceinline__ Fq mul_sub2(const Fq& a, const Fq& b, const Fq& c, const Fq& d) { return fq_mul_sub2(a, b, c, d); }
  static __device__ __forceinline__ Fq add(const Fq& a, const Fq& b) { return fq_add(a, b); }
  static __device__ __forceinline__ Fq sub(const Fq& a, const Fq& b) { return fq_sub(a, b); }
  static __device__ __forceinline__ Fq dbl(const Fq& a) { return fq_dbl(a); }
  static __device__ __forceinline__ Fq neg(const Fq& a) { return fq_neg(a); }
  static __device__ __forceinline__ bool is_zero(const Fq& a) { return fq_is_zero(a); }
};
template <> struct FqOps<true> {
  static __device__ __forceinline__ Fq mul(const Fq& a, const Fq& b) { return fq_mul_lazy(a, b); }
  static __device__ __forceinline__ Fq sqr(const Fq& a) { return fq_sqr_lazy(a); }
  static __device__ __forceinline__ Fq mul_sub2(const Fq& a, const Fq& b, const Fq& c, const Fq& d) { return fq_mul_sub2_lazy(a, b, c, d); }
  static __device__ __forceinline__ Fq add(const Fq& a, const Fq& b) { return fq_add2(a, b); }
  static __device__ __forceinline__ Fq sub(const Fq& a, const Fq& b) { return fq_sub2(a, b); }
  static __device__ __forceinline__ Fq dbl(const Fq& a) { return fq_dbl2(a); }
  static __device__ __forceinline__ Fq neg(const Fq& a) { return fq_neg_lazy(a); }   // a canonical: q - a in [1, q]
  // exact: zero mod q, i.e. 0 or q in [0, 2q)
  static __device__ __forceinline__ bool is_zero(const Fq& a) { return fq_is_zero2(a); }
};

// The identity test ZZ == 0 stays exact on lazy values: ZZ is zeroed only explicitly (xyzz_identity), and every other ZZ
// is a product of factors that are non-zero mod q (the new ZZ of an addition is ZZ1 (ZZ2) PP with PP != 0 mod q, of a
// doubling V ZZ1 with V = 4 Y1^2 != 0: G1 has no point of order 2), which lies in [0, 2q) and is neither 0 nor q.

// 2 * (affine P), P != identity.  P canonical, or y lazy in [1, q] (a negated table point).
template <bool LAZY = false>
static __device__ __noinline__ void xyzz_mdbl(G1Xyzz& r, const G1Affine p) {
  using F = FqOps<LAZY>;
  Fq u = F::dbl(p.y);                  // < 2q (every value below: < 2q)
  Fq v = F::sqr(u);
  Fq w = F::mul(u, v);
  Fq s = F::mul(p.x, v);
  Fq xx = F::sqr(p.x);
  Fq m = F::add(F::dbl(xx), xx);
  Fq x3 = F::sub(F::sqr(m), F::dbl(s));
  r.y = F::mul_sub2(m, F::sub(s, x3), w, p.y);   // m (s - x3) + w (2q - y): < 8 q^2 before the reduction
  r.x = x3;
  r.zz = v;
  r.zzz = w;
}

template <bool LAZY = false>
static __device__ __noinline__ void xyzz_dbl(G1Xyzz& r) {
  using F = FqOps<LAZY>;
  if (xyzz_is_identity(r)) return;
  Fq u = F::dbl(r.y);                  // < 2q (every value below: < 2q)
  Fq v = F::sqr(u);
  Fq w = F::mul(u, v);
  Fq s = F::mul(r.x, v);
  Fq xx = F::sqr(r.x);
  Fq m = F::add(F::dbl(xx), xx);
  Fq x3 = F::sub(F::sqr(m), F::dbl(s));
  Fq y3 = F::mul_sub2(m, F::sub(s, x3), w, r.y);
  r.x = x3;
  r.y = y3;
  r.zz = F::mul(v, r.zz);
  r.zzz = F::mul(w, r.zzz);
}

// acc += P (affine, not identity, canonical); `neg` adds -P.  Handles acc == identity, acc == P, acc == -P.
template <bool LAZY = false>
__device__ __forceinline__ void xyzz_madd(G1Xyzz& acc, const G1Affine& p_in, bool neg) {
  using F = FqOps<LAZY>;
  G1Affine p = p_in;
  if (neg) p.y = F::neg(p.y);          // lazy: q - y in [1, q]
  if (xyzz_is_identity(acc)) {
    acc.x = p.x; acc.y = p.y; acc.zz = fq_one(); acc.zzz = fq_one();
    return;
  }
  Fq u2 = F::mul(p.x, acc.zz);         // < 2q, as every value below
  Fq s2 = F::mul(p.y, acc.zzz);
  Fq pp_ = F::sub(u2, acc.x);
  Fq rr = F::sub(s2, acc.y);
  if (F::is_zero(pp_)) {
    if (F::is_zero(rr)) {
      G1Xyzz d;  // separate object so `acc` itself never has its address taken
      xyzz_mdbl<LAZY>(d, p);
      acc = d;
    } else {
      acc = xyzz_identity();
    }
    return;
  }
  Fq pp = F::sqr(pp_);
  Fq ppp = F::mul(pp_, pp);
  Fq q = F::mul(acc.x, pp);
  Fq x3 = F::sub(F::sub(F::sqr(rr), ppp), F::dbl(q));
  Fq y3 = F::mul_sub2(rr, F::sub(q, x3), acc.y, ppp);   // rr (q - x3) + y1 (2q - ppp): < 8 q^2 before the reduction
  acc.x = x3;
  acc.y = y3;
  acc.zz = F::mul(acc.zz, pp);
  acc.zzz = F::mul(acc.zzz, ppp);
}

// acc += b (both XYZZ), all special cases handled.
template <bool LAZY = false>
static __device__ __noinline__ void xyzz_add(G1Xyzz& acc, const G1Xyzz& b) {
  using F = FqOps<LAZY>;
  if (xyzz_is_identity(b)) return;
  if (xyzz_is_identity(acc)) {
    acc = b;
    return;
  }
  Fq u1 = F::mul(acc.x, b.zz);         // < 2q, as every value below
  Fq u2 = F::mul(b.x, acc.zz);
  Fq s1 = F::mul(acc.y, b.zzz);
  Fq s2 = F::mul(b.y, acc.zzz);
  Fq pp_ = F::sub(u2, u1);
  Fq rr = F::sub(s2, s1);
  if (F::is_zero(pp_)) {
    if (F::is_zero(rr)) {
      xyzz_dbl<LAZY>(acc);
    } else {
      acc = xyzz_identity();
    }
    return;
  }
  Fq pp = F::sqr(pp_);
  Fq ppp = F::mul(pp_, pp);
  Fq q = F::mul(u1, pp);
  Fq x3 = F::sub(F::sub(F::sqr(rr), ppp), F::dbl(q));
  Fq y3 = F::mul_sub2(rr, F::sub(q, x3), s1, ppp);      // < 8 q^2 before the reduction
  acc.x = x3;
  acc.y = y3;
  acc.zz = F::mul(F::mul(acc.zz, b.zz), pp);
  acc.zzz = F::mul(F::mul(acc.zzz, b.zzz), ppp);
}

// acc = k * acc for a small non-negative integer k (double-and-add, MSB first).
template <bool LAZY = false>
static __device__ __noinline__ void xyzz_mul_small(G1Xyzz& acc, uint32_t k) {
  if (k == 0 || xyzz_is_identity(acc)) {
    acc = xyzz_identity();
    return;
  }
  G1Xyzz base = acc;
  int top = 31 - __clz(k);
  for (int b = top - 1; b >= 0; b--) {
    xyzz_dbl<LAZY>(acc);
    if ((k >> b) & 1) xyzz_add<LAZY>(acc, base);
  }
}

// [r]P == identity, r = the group order, MSB-first double-and-add in XYZZ (254 doublings + 131 mixed additions).
static __device__ __noinline__ bool g1_in_subgroup(const G1Affine& p) {
  const uint32_t r[8] = TP_FR_MOD;
  G1Xyzz acc;
  acc.x = p.x;
  acc.y = p.y;
  acc.zz = fq_one();
  acc.zzz = fq_one();
  for (int bit = 253; bit >= 0; bit--) {  // bit 254 is the leading one
    xyzz_dbl(acc);
    if ((r[bit >> 5] >> (bit & 31)) & 1) xyzz_madd(acc, p, false);
  }
  return xyzz_is_identity(acc);
}

// [0, 2q) -> [0, q): the last device step of a lazy point before it leaves the device
__device__ __forceinline__ G1Xyzz xyzz_norm2(const G1Xyzz& a) {
  G1Xyzz r;
  r.x = fq_norm2(a.x); r.y = fq_norm2(a.y); r.zz = fq_norm2(a.zz); r.zzz = fq_norm2(a.zzz);
  return r;
}

}  // namespace tp
