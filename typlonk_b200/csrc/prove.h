// Prover pieces shared by tp_prove (api.cu) and tp_prove_batch (prove_batch.cu): the quotient's coset generators,
// L_0(zeta), the scalars of the linearisation polynomial and the proof's byte layout.  The host algebra between the
// device stages; both drivers take it from here so that their proofs agree byte for byte.
#pragma once
#include "circuit.h"
#include "transcript.h"

namespace tpp {

using tph::HFr;

// g^k, k = 0..3, g = omega_4n: coset k of the 4n domain is g^k H
inline void coset_gens(unsigned log_n, HFr gens[4]) {
  for (unsigned k = 0; k < 4; k++) gens[k] = tp::omega_for_log(log_n + 2).pow_u64(k);
}

// L_0(zeta) = (zeta^n - 1) / (n (zeta - 1)) (utils.rs:150-159)
inline HFr l0_at(const HFr& zeta, size_t n) {
  if (zeta == HFr::one()) return HFr::one();
  return (zeta.pow_u64((uint64_t)n) - HFr::one()) * (HFr::from_u64((uint64_t)n) * (zeta - HFr::one())).inv();
}

// linearisation_poly (proof.rs:376-439): r = constant (at X^0) + sum_j s[j] * poly_j over these polynomials
enum { R_QL, R_QR, R_QO, R_QM, R_QC, R_Z, R_S3, R_T0, R_T1, R_T2, R_TERMS };
struct ProofEvals {
  HFr ev[5];         // a b c z z-omega at zeta (z-omega: at zeta * omega)
  HFr sig_bar[2];    // sigma_1, sigma_2 at zeta
  HFr pi_bar;        // public-input polynomial at zeta
};
// s: R_TERMS scalars, then the constant
inline void lin_scalars(const HFr k[3], const ProofEvals& e, const HFr& alpha, const HFr& beta, const HFr& gamma,
                        const HFr& zeta, size_t n, HFr s[R_TERMS + 1]) {
  const HFr a = e.ev[0], b = e.ev[1], cc = e.ev[2], zw = e.ev[4];
  HFr l2 = HFr::one();
  for (int i = 0; i < 3; i++) l2 = l2 * (e.ev[i] + k[i] * beta * zeta + gamma);
  const HFr perm_ab = (a + beta * e.sig_bar[0] + gamma) * (b + beta * e.sig_bar[1] + gamma);
  const HFr zn = zeta.pow_u64((uint64_t)n);
  const HFr zh = zn - HFr::one();
  const HFr l0 = l0_at(zeta, n);
  const HFr alpha2 = alpha.sqr();
  const HFr ab_zw = alpha * perm_ab * zw;
  s[R_QL] = a;
  s[R_QR] = b;
  s[R_QO] = cc.neg();
  s[R_QM] = a * b;
  s[R_QC] = HFr::one();
  s[R_Z] = alpha * l2 + alpha2 * l0;
  s[R_S3] = (ab_zw * beta).neg();
  s[R_T0] = zh.neg();
  s[R_T1] = (zh * zn).neg();
  s[R_T2] = (zh * zn * zn).neg();
  s[R_TERMS] = e.pi_bar - ab_zw * (gamma + cc) - alpha2 * l0;
}

inline void put_g1(uint8_t*& w, const uint8_t pt[TP_G1_BYTES]) {
  tph::serialize_g1_unchecked(pt, w);
  w += 96;
}
inline void put_fr(uint8_t*& w, const HFr& x) {
  HFr c = x.from_mont();
  memcpy(w, c.v, 32);
  w += 32;
}
// the TP_PROOF_FIXED_BYTES block (proof.rs:85-95): com a b c z, opening witnesses a b c z z-omega r, t commitments
inline void write_proof(uint8_t* w, const uint8_t com[4][TP_G1_BYTES], const uint8_t wit[6][TP_G1_BYTES],
                        const uint8_t tcom[3][TP_G1_BYTES], const HFr ev[5], const HFr& zeta, const HFr& r_bar) {
  for (int i = 0; i < 3; i++) {
    put_g1(w, com[i]);
    put_g1(w, wit[i]);
    put_fr(w, ev[i]);
  }
  put_g1(w, com[3]);
  put_g1(w, wit[3]);
  put_fr(w, ev[3]);
  put_g1(w, wit[4]);
  put_fr(w, ev[4]);
  put_fr(w, zeta);
  for (int i = 0; i < 3; i++) put_g1(w, tcom[i]);
  put_g1(w, wit[5]);
  put_fr(w, r_bar);
}

}  // namespace tpp
