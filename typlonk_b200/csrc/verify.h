// Verifier pieces shared by tp_verify (verify.cu) and tp_verify_batch (verify_batch.cu): proof parsing, the
// Fiat-Shamir challenges, the circuit's verifier values, the scalars of the linearisation commitment and the host half
// of one proof's check.
#pragma once
#include "circuit.h"
#include "pairing.h"

namespace tpv {

using tph::G1Aff;
using tph::HFr;

struct SrsPairing {
  tph::G2Aff g2, g2s;
  tph::G2Prepared pg2, pg2s;
};

struct ParsedProof {  // proof.rs:85-95 in the order tp_prove writes it
  G1Aff com[4];       // a b c z
  G1Aff wit[6];       // a b c z z-omega r
  HFr ev[5];          // a b c z z-omega
  HFr point, r_eval;
  G1Aff t[3];
  uint8_t com_abi[4][TP_G1_BYTES];
};
// false: a coordinate or scalar is not canonical, or a flag is misplaced
bool parse_proof(const uint8_t* p, ParsedProof* o);
bool points_on_curve(const ParsedProof& p);
// verify_challenges (proof.rs:235-244)
void proof_challenges(const ParsedProof& p, HFr* alpha, HFr* beta, HFr* gamma, HFr* point);

struct VerifierValues {
  G1Aff fixed[5], sigma[3], identity;
  HFr k[3], sigma_bar[2], public_eval;
  uint64_t n;
};
// fixed / sigma / identity / k / n of circuit c (the eight commitments: one batched MSM on first use, then cached)
int circuit_verifier_values(tp_ctx* ctx, tp_circuit* c, VerifierValues* v);

// linearisation_commitment (proof.rs:441-503) written as sum_j s[j] * base_j over these bases
enum { LIN_QL, LIN_QR, LIN_QO, LIN_QM, LIN_QC, LIN_Z, LIN_S3, LIN_ID, LIN_T0, LIN_T1, LIN_T2, LIN_TERMS };
// l0 = L_0(zeta) (utils.rs:150-159) is passed in so that a batch can share one inversion
void lin_scalars(const VerifierValues& v, const ParsedProof& p, const HFr& alpha, const HFr& beta, const HFr& gamma,
                 const HFr& l0, HFr s[LIN_TERMS]);
// n (zeta - 1): the denominator of L_0(zeta) when zeta != 1
HFr l0_denominator(uint64_t n, const HFr& zeta);

// proof.rs:195-233 after the device work (sigma_bar and public_eval of v are this proof's)
bool verify_host(const SrsPairing& sp, const VerifierValues& v, const ParsedProof& p);

}  // namespace tpv
