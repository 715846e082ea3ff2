// Proof format v2 (DESIGN.md, "Proof format v2"): the prover's tail after the quotient, the constant-size key, the
// host-only verifier and the proof's wire form.
//
// The stages up to t are v1's (tpp::prove_to_quotient, api.cu) with the v2 transcript as the challenge source and the
// public-input column built from column a.  After t: one MSM batch for [t0] [t1] [t2], then zeta; one batched scan for
// a, b, c, sigma_1, sigma_2 (and PI) at zeta and z at zeta omega with its quotient; r as in v1, then
// P = r + sum_j v^j (p_j - y_j); one opening of P at zeta; one MSM batch of two.
#include "prove.h"
#include "verify.h"

#include <string>

using namespace tp;
using namespace tph;
using namespace tpv;

struct tp_vk2 {
  uint64_t n = 0, ell = 0;
  unsigned log_n = 0;
  HFr k[3];
  G1Aff pts[9];                  // q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 srs[0]
  SrsPairing sp;
  uint8_t wire[TP_VK2_BYTES];
  uint8_t digest[64];            // Blake2b-512 of `wire`: what the transcript binds
};

namespace {

constexpr size_t OFF_N = 8, OFF_L = 16, OFF_K = 24, OFF_G1 = 120, OFF_G2 = 984, OFF_G2S = 1176;
const char* const kG1Names[9] = {"q_l", "q_r", "q_o", "q_m", "q_c", "sigma_1 commitment", "sigma_2 commitment",
                                 "sigma_3 commitment", "srs[0]"};
const char* const kProofG1Names[9] = {"[a]", "[b]", "[c]", "[z]", "[t0]", "[t1]", "[t2]", "W_zeta", "W_zeta_omega"};
constexpr size_t PROOF_G1 = 9, PROOF_FR = 6, PROOF_FR_OFF = 9 * 96;

thread_local std::string g_err;
int host_fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

__global__ void __launch_bounds__(256) k_pi_from_column(const Fr* __restrict__ a, size_t ell, size_t n, Fr* __restrict__ pi) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) pi[i] = i < ell ? fr_neg(a[i]) : fr_zero();
}

void put_u64(uint8_t* w, uint64_t v) {
  for (int i = 0; i < 8; i++) w[i] = (uint8_t)(v >> (8 * i));
}
uint64_t get_u64(const uint8_t* r) {
  uint64_t v = 0;
  for (int i = 7; i >= 0; i--) v = (v << 8) | r[i];
  return v;
}
void abi_of(const G1Aff& p, uint8_t out[TP_G1_BYTES]) {
  memcpy(out, p.x.v, 48);
  memcpy(out + 48, p.y.v, 48);
  out[96] = p.inf ? 1 : 0;
}
bool same_point(const G1Aff& a, const G1Aff& b) { return a.inf == b.inf && (a.inf || (a.x == b.x && a.y == b.y)); }
bool in_g1(const G1Aff& p) { return p.inf || g1_mul_u64limbs(g1_from_aff(p), FR_PARAMS.mod, 4).is_identity(); }

// ark-serialize 0.3 uncompressed G1: canonical coordinates and flags; check 1: + on the curve; 2: + in G1
bool read_point(const uint8_t in[96], int check, G1Aff* out) {
  uint64_t x[6], y[6];
  memcpy(x, in, 48);
  memcpy(y, in + 48, 48);
  if (in[95] & 0x80) return false;
  if (in[95] & 0x40) {
    y[5] &= ~((uint64_t)0x40 << 56);
    for (int i = 0; i < 6; i++)
      if (x[i] != 0 || y[i] != (i == 0 ? 1u : 0u)) return false;
    *out = {HFq::zero(), HFq::one(), true};
    return true;
  }
  if (ge<6>(x, FQ_PARAMS.mod) || ge<6>(y, FQ_PARAMS.mod)) return false;
  *out = {HFq::to_mont(x), HFq::to_mont(y), false};
  if (check >= 1 && !g1aff_on_curve(*out)) return false;
  return check < 2 || in_g1(*out);
}
bool read_scalar(const uint8_t in[32], HFr* out) {
  uint64_t v[4];
  memcpy(v, in, 32);
  if (ge<4>(v, FR_PARAMS.mod)) return false;
  *out = HFr::to_mont(v);
  return true;
}
void write_scalar(uint8_t* w, const HFr& x) {
  HFr c = x.from_mont();
  memcpy(w, c.v, 32);
}

void finish_key(tp_vk2* vk) {
  uint8_t* w = vk->wire;
  memcpy(w, "TPK2", 4);
  const uint32_t version = 1;
  memcpy(w + 4, &version, 4);
  put_u64(w + OFF_N, vk->n);
  put_u64(w + OFF_L, vk->ell);
  for (int i = 0; i < 3; i++) write_scalar(w + OFF_K + 32 * i, vk->k[i]);
  for (int i = 0; i < 9; i++) {
    uint8_t abi[TP_G1_BYTES];
    abi_of(vk->pts[i], abi);
    serialize_g1_unchecked(abi, w + OFF_G1 + 96 * i);
  }
  g2_to_wire(vk->sp.g2, w + OFF_G2);
  g2_to_wire(vk->sp.g2s, w + OFF_G2S);
  Blake2b b;
  b.init();
  b.update(vk->wire, TP_VK2_BYTES);
  b.finalize(vk->digest);
}

struct ChallengesV2 : tpp::ChallengeSource {
  TranscriptV2* tr;
  explicit ChallengesV2(TranscriptV2* t) : tr(t) {}
  void after_abc(const uint8_t com[4][TP_G1_BYTES], HFr* beta, HFr* gamma) override {
    tr->absorb("abc", {com[0], com[1], com[2]});
    *beta = tr->squeeze(0);
    *gamma = tr->squeeze(1);
  }
  void after_z(const uint8_t com[4][TP_G1_BYTES], HFr* alpha) override {
    tr->absorb("z", {com[3]});
    *alpha = tr->squeeze(0);
  }
};

// Everything after the quotient (rounds 3-5 of the prover)
int prove_v2_tail(tp_ctx* ctx, tp_circuit* c, TranscriptV2& tr, const tpp::Round3& st, uint8_t* proof_out) {
  const size_t n = c->n;
  const tp_srs* srs = c->srs;
  uint8_t tcom[3][TP_G1_BYTES];
  {
    const Fr* sets[3] = {c->t, c->t + n, c->t + 2 * n};
    TP_TRY(msm_batch_dev(ctx, srs, sets, 3, n, tcom));
  }
  tr.absorb("t", {tcom[0], tcom[1], tcom[2]});
  const HFr zeta = tr.squeeze(0);
  if (zeta.pow_u64((uint64_t)n) == HFr::one()) return fail(ctx, TP_ERR_ZERO_DENOMINATOR, "prove_v2: zeta^n = 1");
  const HFr omega = omega_for_log(c->log_n);
  // z at zeta omega with its quotient (W_zeta_omega's polynomial), then a b c sigma_1 sigma_2 (PI) at zeta: one scan
  HFr ys[7];
  {
    const Fr* polys[7] = {c->z_coef, c->adv_coef[0], c->adv_coef[1], c->adv_coef[2], c->sig_coef[0], c->sig_coef[1], c->pi_coef};
    Fr* quots[7] = {c->q[0], nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    Fr points[7];
    for (int i = 0; i < 7; i++) points[i] = to_dev(i == 0 ? zeta * omega : zeta);
    TP_TRY(poly_open_batch_dev(ctx, polys, n, points, quots, st.pi_zero ? 6 : 7, ys));
  }
  const HFr ev[6] = {ys[1], ys[2], ys[3], ys[4], ys[5], ys[0]};   // a b c sigma_1 sigma_2 z(zeta omega)
  tr.absorb("evals", {}, ev, 6);
  const HFr v = tr.squeeze(0);
  // r: v1's linearisation with pi_bar = PI(zeta)
  {
    tpp::ProofEvals pe;
    for (int i = 0; i < 3; i++) pe.ev[i] = ev[i];
    pe.ev[3] = HFr::zero();   // z(zeta): not part of r
    pe.ev[4] = ev[5];
    pe.sig_bar[0] = ev[3];
    pe.sig_bar[1] = ev[4];
    pe.pi_bar = st.pi_zero ? HFr::zero() : ys[6];
    HFr s[tpp::R_TERMS + 1];
    tpp::lin_scalars(c->k, pe, st.alpha, st.beta, st.gamma, zeta, n, s);
    const LinTerm terms[tpp::R_TERMS] = {{c->sel_coef[0], 0}, {c->sel_coef[1], 0}, {c->sel_coef[2], 0},
                                         {c->sel_coef[3], 0}, {c->sel_coef[4], 0}, {c->z_coef, 0},
                                         {c->sig_coef[2], 0}, {c->t, 0}, {c->t + n, 0}, {c->t + 2 * n, 0}};
    TP_TRY(lincomb_dev(ctx, terms, tpp::R_TERMS, s, n, 1, c->r, 0));
  }
  // P = r + v (a - a_bar) + v^2 (b - b_bar) + v^3 (c - c_bar) + v^4 (sigma_1 - s1_bar) + v^5 (sigma_2 - s2_bar)
  {
    const LinTerm terms[6] = {{c->r, 0}, {c->adv_coef[0], 0}, {c->adv_coef[1], 0}, {c->adv_coef[2], 0},
                              {c->sig_coef[0], 0}, {c->sig_coef[1], 0}};
    HFr s[7];
    s[0] = HFr::one();
    HFr vj = HFr::one(), cst = HFr::zero();
    for (int j = 1; j <= 5; j++) {
      vj = vj * v;
      s[j] = vj;
      cst = cst - vj * ev[j - 1];
    }
    s[6] = cst;
    TP_TRY(lincomb_dev(ctx, terms, 6, s, n, 1, c->q[1], 0));
  }
  HFr y;
  TP_TRY(poly_open_dev(ctx, c->q[1], n, to_dev(zeta), c->q[2], &y));
  // P(zeta) = r(zeta) = the quotient identity's remainder at zeta: zero for every witness that meets its gates (checked
  // before) and its copy constraints.  One that breaks a copy constraint gets an opening of P - P(zeta), which the
  // verifier (it takes P(zeta) = 0) rejects.
  if (!y.is_zero() && st.z_closes) return fail(ctx, TP_ERR_INTERNAL, "prove_v2: internal error: r(zeta) != 0 for a satisfying witness");
  uint8_t wit[2][TP_G1_BYTES];
  {
    const Fr* sets[2] = {c->q[2], c->q[0]};
    TP_TRY(msm_batch_dev(ctx, srs, sets, 2, n, wit));
  }
  uint8_t* w = proof_out;
  for (int i = 0; i < 4; i++) tpp::put_g1(w, st.com[i]);
  for (int i = 0; i < 3; i++) tpp::put_g1(w, tcom[i]);
  for (int i = 0; i < 2; i++) tpp::put_g1(w, wit[i]);
  for (int i = 0; i < 6; i++) tpp::put_fr(w, ev[i]);
  return TP_OK;
}

// the key's n, cosets, commitments and srs[0] against circuit c's own; once per key (the circuit's commitments and
// srs[0] do not change, and a key is known by its digest)
int key_matches(tp_ctx* ctx, tp_circuit* c, const tp_vk2* vk) {
  if (c->have_v2_key && memcmp(c->v2_key_digest, vk->digest, 64) == 0) return TP_OK;
  VerifierValues v;
  TP_TRY(circuit_verifier_values(ctx, c, &v));
  bool ok = v.n == vk->n && same_point(v.identity, vk->pts[8]);
  for (int i = 0; i < 3; i++) ok &= v.k[i] == vk->k[i];
  for (int i = 0; i < 5; i++) ok &= same_point(v.fixed[i], vk->pts[i]);
  for (int i = 0; i < 3; i++) ok &= same_point(v.sigma[i], vk->pts[5 + i]);
  if (!ok) return fail(ctx, TP_ERR_INVALID_ARG, "prove_v2: the key is not this circuit's");
  memcpy(c->v2_key_digest, vk->digest, 64);
  c->have_v2_key = true;
  return TP_OK;
}

// Rows 0..ell-1 of c are public gates (q_l = 1, every other selector 0) and row ell is not: ell is the number of public
// gates c was traced with.  Reads ell + 1 rows of the five selector columns.
int public_rows_match(tp_ctx* ctx, tp_circuit* c, size_t ell) {
  const size_t rows = ell + 1;   // ell <= n - 3, so row ell exists
  std::vector<HFr> sel(5 * rows);
  for (int k = 0; k < 5; k++)
    TP_CUDA_OK(ctx, cudaMemcpyAsync(sel.data() + k * rows, c->sel_eval[k], rows * sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  auto is_public = [&](size_t j) {
    bool p = sel[j] == HFr::one();
    for (int k = 1; k < 5; k++) p = p && sel[k * rows + j].is_zero();
    return p;
  };
  for (size_t j = 0; j < ell; j++)
    if (!is_public(j)) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: a row below n_public is not a public gate");
  if (is_public(ell)) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: row n_public is a public gate too (n_public is smaller than the circuit's)");
  return TP_OK;
}

int prove_v2_one(tp_ctx* ctx, tp_circuit* c, const tp_vk2* vk, const uint64_t* const advice[3], uint8_t* proof_out) {
  TP_TRY(key_matches(ctx, c, vk));
  std::vector<HFr> pub(vk->ell);
  for (size_t i = 0; i < vk->ell; i++) {
    if (ge<4>(advice[0] + 4 * i, FR_PARAMS.mod)) return fail(ctx, TP_ERR_INVALID_ARG, "prove_v2: public value not reduced modulo r");
    memcpy(pub[i].v, advice[0] + 4 * i, 32);
  }
  TranscriptV2 tr;
  tr.init(vk->digest, pub.data(), pub.size());
  ChallengesV2 ch(&tr);
  return tpp::upload_and_prove(ctx, c, advice, nullptr, 0, [&](const cudaEvent_t* col_ready) {
    tpp::Round3 st;
    TP_TRY(tpp::prove_to_quotient(ctx, c, col_ready, vk->ell, ch, &st));
    return prove_v2_tail(ctx, c, tr, st, proof_out);
  });
}

// L_i(zeta) = omega^i (zeta^n - 1) / (n (zeta - omega^i)), i < count, with one inversion; zeta^n != 1
void lagrange_at(uint64_t n, const HFr& omega, const HFr& zeta, size_t count, std::vector<HFr>* out) {
  std::vector<HFr> den(count), pre(count), wi(count);
  const HFr nn = HFr::from_u64(n), zh = zeta.pow_u64(n) - HFr::one();
  HFr w = HFr::one(), prod = HFr::one();
  for (size_t i = 0; i < count; i++) {
    wi[i] = w;
    den[i] = nn * (zeta - w);
    pre[i] = prod;
    prod = prod * den[i];
    w = w * omega;
  }
  HFr inv = prod.inv();
  out->resize(count);
  for (size_t i = count; i-- > 0;) {
    (*out)[i] = wi[i] * zh * inv * pre[i];
    inv = inv * den[i];
  }
}

}  // namespace

int tpp::pi_from_column_dev(tp_ctx* ctx, const Fr* a, size_t ell, size_t n, Fr* pi) {
  k_pi_from_column<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(a, ell, n, pi);
  TP_LAUNCH(ctx, "k_pi_from_column");
  return TP_OK;
}

extern "C" {

const char* tp_vk2_last_error(void) { return g_err.c_str(); }

int tp_vk2_from_circuit(tp_ctx* ctx, tp_circuit* c, size_t n_public, tp_vk2** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !out) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: null argument");
  if (!ctx->children.empty()) {   // device group: every rank takes part in the commitment MSMs, rank 0's key goes out
    if (c->parts.size() != ctx->children.size()) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: the circuit does not belong to this device group");
    std::vector<tp_vk2*> keys(ctx->children.size(), nullptr);
    int rc = group_run(ctx, [&](tp_ctx* cc, int r) { return tp_vk2_from_circuit(cc, c->parts[r], n_public, &keys[r]); });
    for (size_t r = 1; r < keys.size(); r++) tp_vk2_destroy(keys[r]);
    if (rc != TP_OK) {
      tp_vk2_destroy(keys[0]);
      return rc;
    }
    *out = keys[0];
    return TP_OK;
  }
  if (!c->srs->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: the SRS has no G2 points (tp_srs_set_g2)");
  if (c->n < 4 || n_public > c->n - 3) return fail(ctx, TP_ERR_INVALID_ARG, "vk2_from_circuit: n_public > n - 3");
  TP_TRY(public_rows_match(ctx, c, n_public));
  VerifierValues v;
  TP_TRY(circuit_verifier_values(ctx, c, &v));
  tp_vk2* vk = new tp_vk2();
  vk->n = c->n;
  vk->log_n = c->log_n;
  vk->ell = n_public;
  for (int i = 0; i < 3; i++) vk->k[i] = c->k[i];
  for (int i = 0; i < 5; i++) vk->pts[i] = v.fixed[i];
  for (int i = 0; i < 3; i++) vk->pts[5 + i] = v.sigma[i];
  vk->pts[8] = v.identity;
  vk->sp = *(const SrsPairing*)c->srs->pairing;
  finish_key(vk);
  *out = vk;
  return TP_OK;
}

int tp_vk2_destroy(tp_vk2* vk) {
  delete vk;
  return TP_OK;
}

int tp_vk2_serialize(const tp_vk2* vk, uint8_t* out, size_t cap) {
  if (!vk || !out) return TP_ERR_INVALID_ARG;
  if (cap < TP_VK2_BYTES) return TP_ERR_BUFFER_TOO_SMALL;
  memcpy(out, vk->wire, TP_VK2_BYTES);
  return TP_OK;
}

int tp_vk2_deserialize(const uint8_t* bytes, size_t len, int check, tp_vk2** out) {
  if (!bytes || !out || check < 0 || check > 2) return host_fail(TP_ERR_INVALID_ARG, "vk2_deserialize: null argument or check not in 0..2");
  const char* fn = "vk2_deserialize: ";
  if (len != TP_VK2_BYTES) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "length is not " + std::to_string(TP_VK2_BYTES));
  if (memcmp(bytes, "TPK2", 4) != 0) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "bad tag (not a v2 verification key)");
  uint32_t version;
  memcpy(&version, bytes + 4, 4);
  if (version != 1) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "unsupported version " + std::to_string(version));
  tp_vk2 vk;
  vk.n = get_u64(bytes + OFF_N);
  vk.ell = get_u64(bytes + OFF_L);
  if (vk.n < 4 || (vk.n & (vk.n - 1)) != 0 || vk.n > ((uint64_t)1 << 28))
    return host_fail(TP_ERR_MALFORMED, std::string(fn) + "n = " + std::to_string(vk.n) + " is not a power of two in [4, 2^28]");
  if (vk.ell > vk.n - 3) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "l > n - 3");
  while (((uint64_t)1 << vk.log_n) < vk.n) vk.log_n++;
  for (int i = 0; i < 3; i++)
    if (!read_scalar(bytes + OFF_K + 32 * i, &vk.k[i])) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "k[" + std::to_string(i) + "] not reduced modulo r");
  for (int i = 0; i < 9; i++)
    if (!read_point(bytes + OFF_G1 + 96 * i, check, &vk.pts[i])) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "bad G1 point " + kG1Names[i]);
  if (!g2_from_wire(bytes + OFF_G2, check, &vk.sp.g2) || !g2_on_curve(vk.sp.g2)) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "bad G2 point g2");
  if (!g2_from_wire(bytes + OFF_G2S, check, &vk.sp.g2s) || !g2_on_curve(vk.sp.g2s)) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "bad G2 point g2s");
  vk.sp.pg2 = g2_prepare(vk.sp.g2);
  vk.sp.pg2s = g2_prepare(vk.sp.g2s);
  finish_key(&vk);
  if (memcmp(vk.wire, bytes, TP_VK2_BYTES) != 0) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "not in canonical form");
  *out = new tp_vk2(vk);
  return TP_OK;
}

int tp_prove_v2(tp_ctx* ctx, tp_circuit* c, const tp_vk2* vk, const uint64_t* const advice[3], uint8_t* proof_out,
                size_t proof_cap, uint64_t* public_out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !vk || !proof_out || !advice || !advice[0] || !advice[1] || !advice[2] || (vk->ell && !public_out))
    return fail(ctx, TP_ERR_INVALID_ARG, "prove_v2: null argument");
  if (proof_cap < TP_PROOF_V2_FIXED_BYTES) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "prove_v2: proof buffer too small");
  if (!ctx->children.empty()) {   // every rank proves, rank 0's bytes go out
    if (c->parts.size() != ctx->children.size()) return fail(ctx, TP_ERR_INVALID_ARG, "prove_v2: the circuit does not belong to this device group");
    std::vector<uint8_t> proofs(ctx->children.size() * TP_PROOF_V2_FIXED_BYTES);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) {
      return prove_v2_one(cc, c->parts[r], vk, advice, &proofs[(size_t)r * TP_PROOF_V2_FIXED_BYTES]);
    }));
    memcpy(proof_out, proofs.data(), TP_PROOF_V2_FIXED_BYTES);
  } else {
    TP_TRY(prove_v2_one(ctx, c, vk, advice, proof_out));
  }
  if (vk->ell) memcpy(public_out, advice[0], vk->ell * 32);
  return TP_OK;
}

int tp_verify_v2(const tp_vk2* vk, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
                 size_t n_public, int* ok) {
  if (!vk || !proof || !ok || (n_public && !public_inputs)) return TP_ERR_INVALID_ARG;
  *ok = 0;
  std::vector<HFr> pub(n_public);
  for (size_t i = 0; i < n_public; i++) {
    if (ge<4>(public_inputs + 4 * i, FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
    memcpy(pub[i].v, public_inputs + 4 * i, 32);
  }
  if (proof_len != TP_PROOF_V2_FIXED_BYTES || n_public != vk->ell) return TP_OK;
  G1Aff pt[PROOF_G1];
  uint8_t abi[PROOF_G1][TP_G1_BYTES];
  HFr ev[PROOF_FR];
  for (size_t i = 0; i < PROOF_G1; i++) {
    if (!read_point(proof + 96 * i, 2, &pt[i])) return TP_OK;
    abi_of(pt[i], abi[i]);
  }
  for (size_t i = 0; i < PROOF_FR; i++)
    if (!read_scalar(proof + PROOF_FR_OFF + 32 * i, &ev[i])) return TP_OK;
  TranscriptV2 tr;
  tr.init(vk->digest, pub.data(), n_public);
  tr.absorb("abc", {abi[0], abi[1], abi[2]});
  const HFr beta = tr.squeeze(0), gamma = tr.squeeze(1);
  tr.absorb("z", {abi[3]});
  const HFr alpha = tr.squeeze(0);
  tr.absorb("t", {abi[4], abi[5], abi[6]});
  const HFr zeta = tr.squeeze(0);
  if (zeta.pow_u64(vk->n) == HFr::one()) return TP_OK;
  tr.absorb("evals", {}, ev, PROOF_FR);
  const HFr v = tr.squeeze(0);
  tr.absorb("w", {abi[7], abi[8]});
  const HFr u = tr.squeeze(0);
  const HFr omega = omega_for_log(vk->log_n);
  // PI(zeta) = -sum_{i < l} x_i L_i(zeta)
  HFr pi_bar = HFr::zero();
  if (n_public) {
    std::vector<HFr> lag;
    lagrange_at(vk->n, omega, zeta, n_public, &lag);
    for (size_t i = 0; i < n_public; i++) pi_bar = pi_bar - pub[i] * lag[i];
  }
  tpp::ProofEvals pe;
  for (int i = 0; i < 3; i++) pe.ev[i] = ev[i];
  pe.ev[3] = HFr::zero();
  pe.ev[4] = ev[5];
  pe.sig_bar[0] = ev[3];
  pe.sig_bar[1] = ev[4];
  pe.pi_bar = pi_bar;
  HFr s[tpp::R_TERMS + 1];
  tpp::lin_scalars(vk->k, pe, alpha, beta, gamma, zeta, vk->n, s);
  // rhs = [r] + sum_j v^j [p_j] - (sum_j v^j y_j) G + u [z] - u z_bar_omega G + zeta W_zeta + u zeta omega W_zeta_omega
  const G1Aff* r_bases[tpp::R_TERMS] = {&vk->pts[0], &vk->pts[1], &vk->pts[2], &vk->pts[3], &vk->pts[4],
                                        &pt[3], &vk->pts[7], &pt[4], &pt[5], &pt[6]};
  HG1 rhs = HG1::identity();
  for (int j = 0; j < tpp::R_TERMS; j++) rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(*r_bases[j]), s[j]));
  const G1Aff* opened[5] = {&pt[0], &pt[1], &pt[2], &vk->pts[5], &vk->pts[6]};
  HFr vj = HFr::one(), g_scalar = s[tpp::R_TERMS] - u * ev[5];
  for (int j = 0; j < 5; j++) {
    vj = vj * v;
    rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(*opened[j]), vj));
    g_scalar = g_scalar - vj * ev[j];
  }
  rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(vk->pts[8]), g_scalar));
  rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(pt[3]), u));
  rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(pt[7]), zeta));
  rhs = g1_add(rhs, g1_mul_fr(g1_from_aff(pt[8]), u * zeta * omega));
  const HG1 lhs = g1_add(g1_from_aff(pt[7]), g1_mul_fr(g1_from_aff(pt[8]), u));
  // e(lhs, g2s) * e(-rhs, g2) = 1
  G1Aff ps[2] = {g1_to_aff(lhs), g1_to_aff(g1_neg(rhs))};
  const G2Prepared* qs[2] = {&vk->sp.pg2s, &vk->sp.pg2};
  *ok = pairing_product_is_one(ps, qs, 2) ? 1 : 0;
  return TP_OK;
}

int tp_proof_v2_encode(const uint8_t fixed[TP_PROOF_V2_FIXED_BYTES], const uint64_t* public_inputs, size_t n_public,
                       uint8_t* out, size_t cap, size_t* written) {
  if (!fixed || (n_public && !public_inputs)) return TP_ERR_INVALID_ARG;
  const size_t need = TP_PROOF_V2_FIXED_BYTES + 8 + 32 * n_public;
  if (written) *written = need;
  if (!out || cap < need) return TP_ERR_BUFFER_TOO_SMALL;
  for (size_t i = 0; i < n_public; i++)
    if (ge<4>(public_inputs + 4 * i, FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  memcpy(out, fixed, TP_PROOF_V2_FIXED_BYTES);
  put_u64(out + TP_PROOF_V2_FIXED_BYTES, n_public);
  for (size_t i = 0; i < n_public; i++) {
    HFr x;
    memcpy(x.v, public_inputs + 4 * i, 32);
    write_scalar(out + TP_PROOF_V2_FIXED_BYTES + 8 + 32 * i, x);
  }
  return TP_OK;
}

int tp_proof_v2_decode(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_V2_FIXED_BYTES],
                       uint64_t* public_out, size_t public_cap, size_t* n_public) {
  if (!bytes || !n_public) return host_fail(TP_ERR_INVALID_ARG, "proof_v2_decode: null argument");
  const char* fn = "proof_v2_decode: ";
  if (len < TP_PROOF_V2_FIXED_BYTES + 8) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "truncated");
  const uint64_t l = get_u64(bytes + TP_PROOF_V2_FIXED_BYTES);
  if (l > (len - TP_PROOF_V2_FIXED_BYTES - 8) / 32 || len != TP_PROOF_V2_FIXED_BYTES + 8 + 32 * l)
    return host_fail(TP_ERR_MALFORMED, std::string(fn) + "length does not match the public-value count");
  for (size_t i = 0; i < PROOF_G1; i++) {
    G1Aff p;
    if (!read_point(bytes + 96 * i, 1, &p)) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "bad G1 point " + kProofG1Names[i]);
  }
  std::vector<HFr> vals(l + PROOF_FR);
  for (size_t i = 0; i < PROOF_FR; i++)
    if (!read_scalar(bytes + PROOF_FR_OFF + 32 * i, &vals[i])) return host_fail(TP_ERR_MALFORMED, std::string(fn) + "evaluation not reduced modulo r");
  for (size_t i = 0; i < l; i++)
    if (!read_scalar(bytes + TP_PROOF_V2_FIXED_BYTES + 8 + 32 * i, &vals[PROOF_FR + i]))
      return host_fail(TP_ERR_MALFORMED, std::string(fn) + "public value " + std::to_string(i) + " not reduced modulo r");
  *n_public = l;
  if (fixed_out) memcpy(fixed_out, bytes, TP_PROOF_V2_FIXED_BYTES);
  if (!public_out) return TP_OK;
  if (public_cap < l) return host_fail(TP_ERR_BUFFER_TOO_SMALL, "proof_v2_decode: public-value buffer too small");
  for (size_t i = 0; i < l; i++) memcpy(public_out + 4 * i, vals[PROOF_FR + i].v, 32);
  return TP_OK;
}

}  // extern "C"
