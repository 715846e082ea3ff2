// CompiledCircuit as the library holds it (plonk/src/lib.rs:18-35): device-resident selector / permutation tables and
// the per-proof work buffers, shared by the prover driver (api.cu) and the verifier (verify.cu).
#pragma once
#include "common.cuh"

struct tp_circuit {
  size_t n = 0;
  unsigned log_n = 0;
  const tp_srs* srs = nullptr;
  tp::Fr* sel_coef[5] = {0};
  tp::Fr* sel_eval[5] = {0};
  tp::Fr* sel4[5] = {0};
  tp::Fr* id[3] = {0};
  tp::Fr* sig_eval[3] = {0};
  tp::Fr* sig_coef[3] = {0};
  tp::Fr* sig4[3] = {0};
  tp::Fr* l0_4 = nullptr;
  tph::HFr k[3];
  // per-proof work buffers
  tp::Fr* adv_eval[3] = {0};
  tp::Fr* adv_coef[3] = {0};
  tp::Fr* pi_eval = nullptr;
  tp::Fr* pi_coef = nullptr;
  tp::Fr* z_eval = nullptr;  // n + 1
  tp::Fr* z_coef = nullptr;
  tp::Fr* buf4[6] = {0};     // a4 b4 c4 z4 pi4 num4
  tp::Fr* t = nullptr;       // 3n
  tp::Fr* q[6] = {0};        // opening quotients (a, b, c, z, z-omega, r), n each
  tp::Fr* r = nullptr;       // n
  // true while pi_coef and buf4[4] (the public-input polynomial and its 4n evaluations) are known to hold zeros:
  // a proof whose public inputs are all zero -- the only kind the reference can prove, SURVEY.md App. D.1 -- then
  // skips that polynomial's six transforms
  bool pi_buffers_zero = false;
  std::vector<void*> allocs;
  // tp_prove_batch (prove_batch.cu): the per-proof buffers of `wave_cap` proofs, grown on demand, freed with the circuit
  tp::Fr* wave = nullptr;
  size_t wave_cap = 0;
  std::vector<tp_circuit*> parts;  // circuit of a device group: one per rank (n and log_n are set, nothing else)
  // verifier state (verify.cu): the eight commitments of the circuit itself, computed on first use and kept
  // (the reference recomputes the sigma commitments in every verify, permutation/src/lib.rs:180-194)
  bool have_fixed_com = false, have_sigma_com = false;
  uint8_t fixed_com[5][TP_G1_BYTES];
  uint8_t sigma_com[3][TP_G1_BYTES];
  // tp_prove_v2 (prove_v2.cu): digest of the last v2 key found to be this circuit's, so the check runs once per key
  bool have_v2_key = false;
  uint8_t v2_key_digest[64];
};
