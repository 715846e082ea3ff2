// Verifier: CompiledCircuit::verify (plonk/src/proof.rs:59-63, 195-281), linearisation_commitment (:441-503),
// KzgScheme::verify (kzg/src/lib.rs:66-81), CompiledPermutation::sigma_evals / sigma_commitments
// (permutation/src/lib.rs:165-194), Srs::g2 (kzg/src/srs.rs:25-28).
//
// Split: everything that scales with the circuit runs on the device with the prover's kernels -- the public-input
// interpolation + evaluation, the sigma evaluations at the challenge point (from the cached coefficient forms; the
// reference re-interpolates all three per call) and the eight circuit commitments (MSM, once per circuit; the
// reference recomputes the sigma ones per call).  What is left is O(1): two hashes, ~20 G1 scalar multiplications and
// the pairings (pairing.h), done by the calling thread.
#include "verify.h"
#include "transcript.h"

#include <future>
#include <system_error>

using namespace tp;
using namespace tph;
using namespace tpv;

namespace {

// ark-serialize 0.3 uncompressed, unchecked G1 (x | y canonical LE, infinity = bit 6 of the last byte)
bool read_g1(const uint8_t in[96], G1Aff* out) {
  uint64_t x[6], y[6];
  memcpy(x, in, 48);
  memcpy(y, in + 48, 48);
  if (in[95] & 0x80) return false;  // the compressed form's sign flag has no place in an uncompressed record
  if (in[95] & 0x40) {              // infinity: canonical only as (x, y) = (0, 1) | flag
    y[5] &= ~((uint64_t)0x40 << 56);
    for (int i = 0; i < 6; i++)
      if (x[i] != 0 || y[i] != (i == 0 ? 1u : 0u)) return false;
    *out = {HFq::zero(), HFq::one(), true};
    return true;
  }
  if (ge<6>(x, FQ_PARAMS.mod) || ge<6>(y, FQ_PARAMS.mod)) return false;
  *out = {HFq::to_mont(x), HFq::to_mont(y), false};
  return true;
}
bool read_fr(const uint8_t in[32], HFr* out) {
  uint64_t v[4];
  memcpy(v, in, 32);
  if (ge<4>(v, FR_PARAMS.mod)) return false;
  *out = HFr::to_mont(v);
  return true;
}
void abi_g1(const G1Aff& p, uint8_t out[TP_G1_BYTES]) {
  memcpy(out, p.x.v, 48);
  memcpy(out + 48, p.y.v, 48);
  out[96] = p.inf ? 1 : 0;
}

}  // namespace

namespace tpv {

bool parse_proof(const uint8_t* p, ParsedProof* o) {
  bool ok = true;
  for (int i = 0; i < 3; i++) {
    ok &= read_g1(p, &o->com[i]) && read_g1(p + 96, &o->wit[i]) && read_fr(p + 192, &o->ev[i]);
    p += 224;
  }
  ok &= read_g1(p, &o->com[3]) && read_g1(p + 96, &o->wit[3]) && read_fr(p + 192, &o->ev[3]);
  p += 224;
  ok &= read_g1(p, &o->wit[4]) && read_fr(p + 96, &o->ev[4]);
  p += 128;
  ok &= read_fr(p, &o->point);
  p += 32;
  for (int i = 0; i < 3; i++) {
    ok &= read_g1(p, &o->t[i]);
    p += 96;
  }
  ok &= read_g1(p, &o->wit[5]) && read_fr(p + 96, &o->r_eval);
  if (ok)
    for (int i = 0; i < 4; i++) abi_g1(o->com[i], o->com_abi[i]);
  return ok;
}
bool points_on_curve(const ParsedProof& p) {
  bool ok = true;
  for (auto& g : p.com) ok &= g1aff_on_curve(g);
  for (auto& g : p.wit) ok &= g1aff_on_curve(g);
  for (auto& g : p.t) ok &= g1aff_on_curve(g);
  return ok;
}
// verify_challenges (proof.rs:235-244)
void proof_challenges(const ParsedProof& p, HFr* alpha, HFr* beta, HFr* gamma, HFr* point) {
  challenges2({p.com_abi[0], p.com_abi[1], p.com_abi[2]}, beta, gamma);
  challenges2({p.com_abi[0], p.com_abi[1], p.com_abi[2], p.com_abi[3]}, alpha, point);
}

}  // namespace tpv

namespace {

// kzg/src/lib.rs:66-81 as one two-pair product over the prepared SRS points
bool kzg_check(const SrsPairing& sp, const G1Aff& identity, const G1Aff& com, const G1Aff& w, const HFr& y, const HFr& z) {
  HG1 b = g1_add(g1_from_aff(com), g1_neg(g1_mul_fr(g1_from_aff(identity), y)));  // C - y G
  HG1 s = g1_add(g1_mul_fr(g1_from_aff(w), z), b);
  G1Aff ps[2] = {w, g1_to_aff(g1_neg(s))};
  const G2Prepared* qs[2] = {&sp.pg2s, &sp.pg2};
  return pairing_product_is_one(ps, qs, 2);
}

}  // namespace

namespace tpv {

// proof.rs:195-233 after the device work.  KzgScheme::verify subtracts y times the prime-subgroup generator (lib.rs:77);
// linearisation_commitment scales `identity()` = commit(1) = srs[0] (lib.rs:82-85) -- the same point for any SRS made
// by Srs::from_secret, kept apart here as in the reference.
bool verify_host(const SrsPairing& sp, const VerifierValues& v, const ParsedProof& p) {
  HFr alpha, beta, gamma, point;
  proof_challenges(p, &alpha, &beta, &gamma, &point);
  if (p.point != point) return false;  // proof.rs:211-213
  const HFr zeta = point;
  const G1Aff gen = {HFq::to_mont(G1_GEN_X), HFq::to_mont(G1_GEN_Y), false};
  unsigned log_n = 0;
  while (((uint64_t)1 << log_n) < v.n) log_n++;
  HFr omega = omega_for_log(log_n);
  // verify_openings (proof.rs:245-281).  The five checks are independent of each other and of the linearisation
  // commitment below (each is two scalar multiplications, a two-pair Miller loop and a final exponentiation of pure
  // host arithmetic), so they run on their own threads while this one assembles the commitment.
  const HFr zeta_omega = zeta * omega;
  std::future<bool> openings[5];
  for (int i = 0; i < 5; i++) {
    const G1Aff* com = &p.com[i < 3 ? i : 3];
    const HFr* at = i == 4 ? &zeta_omega : &zeta;
    auto one = [&sp, &gen, &p, com, at, i] { return kzg_check(sp, gen, *com, p.wit[i], p.ev[i], *at); };
    try {
      openings[i] = std::async(std::launch::async, one);
    } catch (const std::system_error&) {  // no thread to be had: deferred = evaluated by get() on this thread
      openings[i] = std::async(std::launch::deferred, one);
    }
  }
  auto openings_ok = [&openings] {
    bool ok = true;
    for (auto& f : openings) ok &= f.get();
    return ok;
  };
  // linearisation_commitment (proof.rs:441-503)
  HFr zh = zeta.pow_u64(v.n) - HFr::one();
  HFr l0 = zeta == HFr::one() ? HFr::one() : zh * l0_denominator(v.n, zeta).inv();  // utils.rs:150-159
  HFr s[LIN_TERMS];
  lin_scalars(v, p, alpha, beta, gamma, l0, s);
  const G1Aff* bases[LIN_TERMS] = {&v.fixed[0], &v.fixed[1], &v.fixed[2], &v.fixed[3], &v.fixed[4], &p.com[3],
                                   &v.sigma[2], &v.identity, &p.t[0], &p.t[1], &p.t[2]};
  HG1 r = HG1::identity();
  for (int j = 0; j < LIN_TERMS; j++)
    r = g1_add(r, j == LIN_QC ? g1_from_aff(*bases[j]) : g1_mul_fr(g1_from_aff(*bases[j]), s[j]));  // s[LIN_QC] = 1
  bool open_valid = kzg_check(sp, gen, g1_to_aff(r), p.wit[5], p.r_eval, zeta);
  return openings_ok() && open_valid && p.r_eval.is_zero();
}

HFr l0_denominator(uint64_t n, const HFr& zeta) { return HFr::from_u64(n) * (zeta - HFr::one()); }

// proof.rs:441-503: line1 = a q_l + b q_r - c q_o + ab q_m + q_c, line2 = (l2 alpha + l0 alpha^2) z,
// line3 = l3 alpha beta zw sigma_3, line5 = zh (t0 + zeta^n t1 + zeta^2n t2) (utils.rs:110-126),
// r = line1 + line2 - line3 - constant identity - line5
void lin_scalars(const VerifierValues& v, const ParsedProof& p, const HFr& alpha, const HFr& beta, const HFr& gamma,
                 const HFr& l0, HFr s[LIN_TERMS]) {
  const HFr zeta = p.point;
  const HFr a = p.ev[0], b = p.ev[1], c = p.ev[2], zw = p.ev[4];
  const HFr zero = HFr::zero();
  s[LIN_QL] = a;
  s[LIN_QR] = b;
  s[LIN_QO] = zero - c;
  s[LIN_QM] = a * b;
  s[LIN_QC] = HFr::one();
  HFr l2 = HFr::one();
  for (int i = 0; i < 3; i++) l2 = l2 * (p.ev[i] + beta * v.k[i] * zeta + gamma);
  HFr zn = zeta.pow_u64(v.n), zh = zn - HFr::one();
  HFr alpha2 = alpha.sqr();
  s[LIN_Z] = l2 * alpha + l0 * alpha2;
  HFr l3 = (a + beta * v.sigma_bar[0] + gamma) * (b + beta * v.sigma_bar[1] + gamma);
  s[LIN_S3] = zero - l3 * alpha * beta * zw;
  HFr constant = alpha * (l3 * (c + gamma) * zw) + l0 * alpha2 + v.public_eval;
  s[LIN_ID] = zero - constant;
  s[LIN_T0] = zero - zh;
  s[LIN_T1] = zero - zh * zn;
  s[LIN_T2] = zero - zh * zn * zn;
}

int circuit_verifier_values(tp_ctx* ctx, tp_circuit* c, VerifierValues* v) {
  // the circuit's own commitments: one batched MSM the first time
  if (!c->have_fixed_com || !c->have_sigma_com) {
    const Fr* sets[8] = {c->sel_coef[0], c->sel_coef[1], c->sel_coef[2], c->sel_coef[3], c->sel_coef[4],
                         c->sig_coef[0], c->sig_coef[1], c->sig_coef[2]};
    uint8_t outs[8][TP_G1_BYTES];
    TP_TRY(msm_batch_dev(ctx, c->srs, sets, 8, c->n, outs));
    memcpy(c->fixed_com, outs, sizeof(c->fixed_com));
    memcpy(c->sigma_com, outs + 5, sizeof(c->sigma_com));
    c->have_fixed_com = c->have_sigma_com = true;
  }
  for (int i = 0; i < 5; i++) v->fixed[i] = g1aff_decode(c->fixed_com[i]);
  for (int i = 0; i < 3; i++) v->sigma[i] = g1aff_decode(c->sigma_com[i]);
  for (int i = 0; i < 3; i++) v->k[i] = c->k[i];
  {
    uint8_t first[96];
    TP_CUDA_OK(ctx, cudaMemcpyAsync(first, c->srs->g1, 96, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    bool inf = true;
    for (int i = 0; i < 96; i++) inf &= first[i] == 0;
    memcpy(v->identity.x.v, first, 48);
    memcpy(v->identity.y.v, first + 48, 48);
    v->identity.inf = inf;
    if (inf) v->identity = {HFq::zero(), HFq::one(), true};
  }
  v->n = c->n;
  return TP_OK;
}

int circuit_view(tp_ctx* ctx, tp_circuit* c, VerifierView* view) {
  TP_TRY(circuit_verifier_values(ctx, c, &view->v));
  view->log_n = c->log_n;
  memcpy(view->com, c->fixed_com, sizeof(c->fixed_com));
  memcpy(view->com + 5, c->sigma_com, sizeof(c->sigma_com));
  view->sig_coef[0] = c->sig_coef[0];
  view->sig_coef[1] = c->sig_coef[1];
  view->sp = (const SrsPairing*)c->srs->pairing;
  // the prover's public-input buffers
  view->pi_scratch = [c](Fr** eval, Fr** coef) -> int {
    c->pi_buffers_zero = false;
    *eval = c->pi_eval;
    *coef = c->pi_coef;
    return TP_OK;
  };
  return TP_OK;
}

int verify_single(tp_ctx* ctx, size_t n, bool have_g2, const std::function<int(VerifierView*)>& make_view,
                  const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs, size_t n_public, int* ok) {
  if (proof_len < TP_PROOF_FIXED_BYTES) return fail(ctx, TP_ERR_INVALID_ARG, "verify: proof shorter than the fixed block");
  if (!have_g2) return fail(ctx, TP_ERR_INVALID_ARG, "verify: the SRS has no G2 points (tp_srs_set_g2)");
  *ok = 0;
  // the same bound the prover enforces (prove_from_host); Montgomery limbs must be reduced
  if (n_public > n) return fail(ctx, TP_ERR_INVALID_ARG, "verify: more public inputs than rows");
  bool pi_zero = true;
  for (size_t i = 0; i < n_public; i++) {
    if (ge<4>(public_inputs + 4 * i, FR_PARAMS.mod)) return fail(ctx, TP_ERR_INVALID_ARG, "verify: public input not reduced modulo r");
    for (int j = 0; j < 4; j++) pi_zero &= public_inputs[4 * i + j] == 0;
  }
  ParsedProof p;
  if (!parse_proof(proof, &p)) return fail(ctx, TP_ERR_INVALID_ARG, "verify: non-canonical field element in the proof");
  if (!points_on_curve(p)) return TP_OK;
  VerifierView view;
  TP_TRY(make_view(&view));
  VerifierValues& v = view.v;
  // sigma_1, sigma_2 and the public inputs resized to n (proof.rs:204-205), interpolated, at the proof's point (the
  // point is checked against the re-derived challenge on the host side; a mismatch rejects before these are used).
  // All-zero public inputs give PI = 0 without device work.
  {
    const Fr* polys[3] = {view.sig_coef[0], view.sig_coef[1], nullptr};
    Fr* quots[3] = {nullptr, nullptr, nullptr};
    Fr points[3] = {to_dev(p.point), to_dev(p.point), to_dev(p.point)};
    HFr ys[3];
    v.public_eval = HFr::zero();
    if (!pi_zero) {
      Fr *eval, *coef;
      TP_TRY(view.pi_scratch(&eval, &coef));
      TP_CUDA_OK(ctx, cudaMemsetAsync(eval, 0, n * sizeof(Fr), ctx->stream));
      TP_CUDA_OK(ctx, cudaMemcpyAsync(eval, public_inputs, n_public * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
      TP_TRY(ntt_dev(ctx, eval, coef, view.log_n, true, nullptr));
      polys[2] = coef;
    }
    TP_TRY(poly_open_batch_dev(ctx, polys, n, points, quots, pi_zero ? 2 : 3, ys));
    v.sigma_bar[0] = ys[0];
    v.sigma_bar[1] = ys[1];
    if (!pi_zero) v.public_eval = ys[2];
  }
  *ok = verify_host(*view.sp, v, p) ? 1 : 0;
  return TP_OK;
}

}  // namespace tpv

namespace {

int prepare_pairing(const uint8_t g2[TP_G2_BYTES], const uint8_t g2s[TP_G2_BYTES], SrsPairing* sp) {
  sp->g2 = g2_decode(g2);
  sp->g2s = g2_decode(g2s);
  if (!g2_on_curve(sp->g2) || !g2_on_curve(sp->g2s)) return TP_ERR_INVALID_ARG;
  sp->pg2 = g2_prepare(sp->g2);
  sp->pg2s = g2_prepare(sp->g2s);
  return TP_OK;
}

}  // namespace

namespace tp {
int srs_pairing_from_secret(tp_srs* srs, const HFr& tau) {
  srs_pairing_free(srs);
  SrsPairing* sp = new SrsPairing();
  sp->g2 = g2_generator();
  HFr t = tau.from_mont();
  sp->g2s = g2_mul(sp->g2, t.v, 4);
  sp->pg2 = g2_prepare(sp->g2);
  sp->pg2s = g2_prepare(sp->g2s);
  srs->pairing = sp;
  return TP_OK;
}
void srs_pairing_free(tp_srs* srs) {
  delete (SrsPairing*)srs->pairing;
  srs->pairing = nullptr;
}
}  // namespace tp

extern "C" {

int tp_srs_g2(const tp_srs* srs, uint8_t g2[TP_G2_BYTES], uint8_t g2s[TP_G2_BYTES]) {
  if (srs && !srs->parts.empty()) return tp_srs_g2(srs->parts[0], g2, g2s);   // SRS of a device group: every rank holds the same
  if (!srs || !srs->pairing || !g2 || !g2s) return TP_ERR_INVALID_ARG;
  const SrsPairing* sp = (const SrsPairing*)srs->pairing;
  g2_encode(sp->g2, g2);
  g2_encode(sp->g2s, g2s);
  return TP_OK;
}
int tp_srs_set_g2(tp_srs* srs, const uint8_t g2[TP_G2_BYTES], const uint8_t g2s[TP_G2_BYTES]) {
  if (!srs || !g2 || !g2s) return TP_ERR_INVALID_ARG;
  if (!srs->parts.empty()) {
    for (tp_srs* part : srs->parts) TP_TRY(tp_srs_set_g2(part, g2, g2s));
    return TP_OK;
  }
  SrsPairing* sp = new SrsPairing();
  int rc = prepare_pairing(g2, g2s, sp);
  if (rc != TP_OK) {
    delete sp;
    return rc;
  }
  srs_pairing_free(srs);
  srs->pairing = sp;
  return TP_OK;
}

int tp_pairing_check(const uint8_t* g1, const uint8_t* g2, size_t count, int* ok) {
  if (!ok || (count && (!g1 || !g2)) || count > 1024) return TP_ERR_INVALID_ARG;
  std::vector<G1Aff> ps(count);
  std::vector<G2Prepared> prep(count);
  std::vector<const G2Prepared*> qs(count);
  *ok = 0;
  for (size_t i = 0; i < count; i++) {
    ps[i] = g1aff_decode(g1 + i * TP_G1_BYTES);
    G2Aff q = g2_decode(g2 + i * TP_G2_BYTES);
    if (!g1aff_on_curve(ps[i]) || !g2_on_curve(q)) return TP_OK;
    prep[i] = g2_prepare(q);
    qs[i] = &prep[i];
  }
  *ok = pairing_product_is_one(ps.data(), qs.data(), (int)count) ? 1 : 0;
  return TP_OK;
}

int tp_kzg_verify(const uint8_t g2[TP_G2_BYTES], const uint8_t g2s[TP_G2_BYTES], const uint8_t commitment[TP_G1_BYTES],
                  const uint8_t w[TP_G1_BYTES], const uint64_t y[4], const uint64_t z[4], int* ok) {
  if (!g2 || !g2s || !commitment || !w || !y || !z || !ok) return TP_ERR_INVALID_ARG;
  *ok = 0;
  SrsPairing sp;
  TP_TRY(prepare_pairing(g2, g2s, &sp));
  G1Aff c = g1aff_decode(commitment), wp = g1aff_decode(w);
  if (!g1aff_on_curve(c) || !g1aff_on_curve(wp)) return TP_OK;
  HFr yy, zz;
  memcpy(yy.v, y, 32);
  memcpy(zz.v, z, 32);
  const G1Aff gen = {HFq::to_mont(G1_GEN_X), HFq::to_mont(G1_GEN_Y), false};
  *ok = kzg_check(sp, gen, c, wp, yy, zz) ? 1 : 0;
  return TP_OK;
}

int tp_proof_challenges(const uint8_t* proof, size_t proof_len, uint64_t alpha[4], uint64_t beta[4], uint64_t gamma[4],
                        uint64_t point[4]) {
  if (!proof || proof_len < TP_PROOF_FIXED_BYTES) return TP_ERR_INVALID_ARG;
  ParsedProof p;
  if (!parse_proof(proof, &p)) return TP_ERR_INVALID_ARG;
  HFr a, b, g, z;
  proof_challenges(p, &a, &b, &g, &z);
  memcpy(alpha, a.v, 32);
  memcpy(beta, b.v, 32);
  memcpy(gamma, g.v, 32);
  memcpy(point, z.v, 32);
  return TP_OK;
}

int tp_verify_prepared(const tp_verifier_inputs* in, const uint8_t* proof, size_t proof_len, int* ok) {
  if (!in || !proof || !ok || proof_len < TP_PROOF_FIXED_BYTES) return TP_ERR_INVALID_ARG;
  if (in->n < 2 || (in->n & (in->n - 1)) != 0 || in->n > ((uint64_t)1 << 32)) return TP_ERR_INVALID_ARG;
  *ok = 0;
  ParsedProof p;
  if (!parse_proof(proof, &p)) return TP_ERR_INVALID_ARG;
  SrsPairing sp;
  TP_TRY(prepare_pairing(in->g2, in->g2s, &sp));
  VerifierValues v;
  bool on = points_on_curve(p);
  for (int i = 0; i < 5; i++) on &= g1aff_on_curve(v.fixed[i] = g1aff_decode(in->fixed_commitments[i]));
  for (int i = 0; i < 3; i++) on &= g1aff_on_curve(v.sigma[i] = g1aff_decode(in->sigma_commitments[i]));
  on &= g1aff_on_curve(v.identity = g1aff_decode(in->identity));
  if (!on) return TP_OK;
  for (int i = 0; i < 3; i++)
    if (ge<4>(in->cosets[i], FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  for (int i = 0; i < 2; i++)
    if (ge<4>(in->sigma_evals[i], FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  if (ge<4>(in->public_eval, FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  for (int i = 0; i < 3; i++) memcpy(v.k[i].v, in->cosets[i], 32);
  for (int i = 0; i < 2; i++) memcpy(v.sigma_bar[i].v, in->sigma_evals[i], 32);
  memcpy(v.public_eval.v, in->public_eval, 32);
  v.n = in->n;
  *ok = verify_host(sp, v, p) ? 1 : 0;
  return TP_OK;
}

int tp_verify(tp_ctx* ctx, tp_circuit* c, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
              size_t n_public, int* ok) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !proof || !ok || (n_public && !public_inputs)) return fail(ctx, TP_ERR_INVALID_ARG, "verify: null argument");
  if (!ctx->children.empty()) {   // device group: the first call's commitment MSMs are sharded, so every rank takes part
    std::vector<int> oks(ctx->children.size(), 0);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) { return tp_verify(cc, c->parts[r], proof, proof_len, public_inputs, n_public, &oks[r]); }));
    *ok = oks[0];
    return TP_OK;
  }
  return verify_single(ctx, c->n, c->srs->pairing != nullptr, [&](VerifierView* view) { return circuit_view(ctx, c, view); },
                       proof, proof_len, public_inputs, n_public, ok);
}

}  // extern "C"
