// Verifier pieces shared by tp_verify (verify.cu) and tp_verify_batch (verify_batch.cu): proof parsing, the
// Fiat-Shamir challenges, the circuit's verifier values, the scalars of the linearisation commitment and the host half
// of one proof's check.
#pragma once
#include <functional>

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

// Everything the device half of the verifier reads, built from a circuit (circuit_view) or from a verification key
// (verify_key.cu), so that both run the same code.
struct VerifierView {
  VerifierValues v;                 // fixed / sigma / identity / k / n (sigma_bar and public_eval are per proof)
  unsigned log_n;
  uint8_t com[8][TP_G1_BYTES];      // q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 as ABI records
  const tp::Fr* sig_coef[2];        // sigma_1, sigma_2 coefficients on the device, n each
  const SrsPairing* sp;
  // two n-Fr device buffers for PI(zeta) (pad, interpolate, evaluate); asked for only when a public input is non-zero
  std::function<int(tp::Fr** eval, tp::Fr** coef)> pi_scratch;
};
int circuit_view(tp_ctx* ctx, tp_circuit* c, VerifierView* view);

// tp_verify after a device group's fan-out: argument checks, parsing, then the device evaluations and verify_host over
// the view (made only once the proof has parsed and its points are on the curve).
int verify_single(tp_ctx* ctx, size_t n, bool have_g2, const std::function<int(VerifierView*)>& make_view,
                  const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs, size_t n_public, int* ok);

// tp_verify_batch over several views: proof k is checked against views[view_of[k]] (view_of NULL: every proof against
// views[0]).  keys_hash: the rho of tp_vk_verify_batch (keys-v1 tag, every key bound) instead of tp_verify_batch's.
int verify_batch_views(tp_ctx* ctx, const VerifierView* views, size_t n_views, const uint32_t* view_of, bool keys_hash,
                       const uint8_t* proofs, size_t count, const uint64_t* const* public_inputs, const size_t* n_public,
                       int* all_ok, int* each_ok);

}  // namespace tpv

namespace tp {
// wire.cu: G2 records of the ark-serialize 0.3 uncompressed encoding (check as tp_srs_deserialize)
void g2_to_wire(const tph::G2Aff& p, uint8_t out[TP_WIRE_G2_BYTES]);
bool g2_from_wire(const uint8_t in[TP_WIRE_G2_BYTES], int check, tph::G2Aff* out);
}  // namespace tp
