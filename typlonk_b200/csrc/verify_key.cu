// Verification keys: what verify() (proof.rs:195-233, 441-503) reads of a compiled circuit, without the prover's state.
//
// verify() evaluates sigma_1 and sigma_2 at the proof's challenge point (proof.rs:458-459) -- the proof does not carry
// them -- so a key holds both polynomials in coefficient form, 2n Fr on the device (64n bytes on the wire).  Everything
// else is O(1): n, the coset representatives k, the five selector and three sigma commitments, srs[0] (the point the
// linearisation commitment scales) and the SRS's two G2 points.  Verification runs verify.cu's and verify_batch.cu's
// code over a VerifierView built from the key, exactly as tp_verify / tp_verify_batch do from a circuit.
//
// Wire form (ark-serialize 0.3 uncompressed items, our framing):
//   "TPVK" | u32 version = 1 | u64 n | 3 x Fr k | 9 x G1 (q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 identity) |
//   G2 g2 | G2 g2s | Vec<Fr> sigma_1 | Vec<Fr> sigma_2            = 1376 + 64 n bytes
// The sigma scalars are converted out of / into Montgomery form and checked on the device (k_fr_to_wire /
// k_fr_from_wire, wire.cu); the nine G1 points are checked on the host, their subgroup check on the device.
#include "verify.h"
#include "transcript.h"

using namespace tp;
using namespace tph;
using namespace tpv;

struct tp_vk {
  tp_ctx* ctx = nullptr;   // the context the key was made on (a device group's front for a group key)
  size_t n = 0;
  unsigned log_n = 0;
  HFr k[3];
  uint8_t com[8][TP_G1_BYTES];   // q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 (ABI records)
  G1Aff identity;
  SrsPairing sp;
  Fr* sig = nullptr;       // sigma_1 | sigma_2 coefficients, 2n
  Fr* pi = nullptr;        // public-input scratch (evaluations | coefficients, 2n), allocated on first use
  std::vector<tp_vk*> parts;   // key of a device group: one per rank
};

namespace {

constexpr size_t VK_HEAD = 1376;   // everything but the 64n bytes of sigma_1, sigma_2
constexpr size_t OFF_N = 8, OFF_K = 16, OFF_G1 = 112, OFF_G2 = 976, OFF_G2S = 1168, OFF_SIG = 1360;
const char* const kG1Names[9] = {"q_l", "q_r", "q_o", "q_m", "q_c", "sigma_1 commitment", "sigma_2 commitment",
                                 "sigma_3 commitment", "identity"};

int vk_fail(tp_ctx* ctx, int code, const char* fn, const std::string& msg) {
  ctx->err = std::string(fn) + ": " + msg;
  return code;
}

void free_key(tp_vk* vk) {
  if (vk->sig) cudaFree(vk->sig);
  if (vk->pi) cudaFree(vk->pi);
  delete vk;
}

int alloc_sig(tp_ctx* ctx, tp_vk* vk, const char* fn) {
  if (cudaMalloc(&vk->sig, 2 * vk->n * sizeof(Fr)) != cudaSuccess) {
    cudaGetLastError();
    vk->sig = nullptr;
    return vk_fail(ctx, TP_ERR_CUDA, fn, "out of device memory");
  }
  return TP_OK;
}

// A device group front over parts made by `make(rank context, rank, &part)` on every rank.
int group_key(tp_ctx* g, size_t n, tp_vk** out, const std::function<int(tp_ctx*, int, tp_vk**)>& make) {
  tp_vk* front = new tp_vk();
  front->ctx = g;
  front->parts.assign(g->children.size(), nullptr);
  int rc = group_run(g, [&](tp_ctx* c, int r) { return make(c, r, &front->parts[r]); });
  if (rc != TP_OK) {
    group_run(g, [&](tp_ctx* c, int r) { return tp_vk_destroy(c, front->parts[r]); });
    delete front;
    return rc;
  }
  front->n = n ? n : front->parts[0]->n;
  front->log_n = front->parts[0]->log_n;
  *out = front;
  return TP_OK;
}

void key_view(tp_ctx* ctx, tp_vk* vk, VerifierView* view) {
  VerifierValues& v = view->v;
  for (int i = 0; i < 5; i++) v.fixed[i] = g1aff_decode(vk->com[i]);
  for (int i = 0; i < 3; i++) v.sigma[i] = g1aff_decode(vk->com[5 + i]);
  v.identity = vk->identity;
  for (int i = 0; i < 3; i++) v.k[i] = vk->k[i];
  v.n = vk->n;
  view->log_n = vk->log_n;
  memcpy(view->com, vk->com, sizeof(vk->com));
  view->sig_coef[0] = vk->sig;
  view->sig_coef[1] = vk->sig + vk->n;
  view->sp = &vk->sp;
  view->pi_scratch = [ctx, vk](Fr** eval, Fr** coef) -> int {
    if (!vk->pi && cudaMalloc(&vk->pi, 2 * vk->n * sizeof(Fr)) != cudaSuccess) {
      cudaGetLastError();
      vk->pi = nullptr;
      return fail(ctx, TP_ERR_CUDA, "vk_verify: out of device memory");
    }
    *eval = vk->pi;
    *coef = vk->pi + vk->n;
    return TP_OK;
  };
}

// ark-serialize 0.3 uncompressed G1 -> ABI record; check >= 1 adds "on the curve".  false: not canonical / bad flags.
bool g1_record(const uint8_t in[TP_WIRE_G1_BYTES], int check, uint8_t abi[TP_G1_BYTES]) {
  uint64_t x[6], y[6];
  memcpy(x, in, 48);
  memcpy(y, in + 48, 48);
  const uint8_t flags = in[95] & 0xc0;
  y[5] &= ~((uint64_t)0xc0 << 56);
  if (flags & 0x80) return false;
  if (flags & 0x40) {   // infinity: canonical only as (0, 1)
    for (int i = 0; i < 6; i++)
      if (x[i] != 0 || y[i] != (i == 0 ? 1u : 0u)) return false;
    memset(abi, 0, TP_G1_BYTES);
    abi[96] = 1;
    return true;
  }
  if (ge<6>(x, FQ_PARAMS.mod) || ge<6>(y, FQ_PARAMS.mod)) return false;
  G1Aff p = {HFq::to_mont(x), HFq::to_mont(y), false};
  if (check >= 1 && !g1aff_on_curve(p)) return false;
  memcpy(abi, p.x.v, 48);
  memcpy(abi + 48, p.y.v, 48);
  abi[96] = 0;
  return true;
}

int deserialize_one(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_vk** out) {
  const char* fn = "vk_deserialize";
  if (len < VK_HEAD) return vk_fail(ctx, TP_ERR_MALFORMED, fn, "truncated");
  if (memcmp(bytes, "TPVK", 4) != 0) return vk_fail(ctx, TP_ERR_MALFORMED, fn, "bad tag (not a verification key)");
  uint32_t version;
  memcpy(&version, bytes + 4, 4);
  if (version != 1) return vk_fail(ctx, TP_ERR_MALFORMED, fn, "unsupported version " + std::to_string(version));
  uint64_t n;
  memcpy(&n, bytes + OFF_N, 8);
  if (n < 2 || (n & (n - 1)) != 0 || n > ((uint64_t)1 << 28))
    return vk_fail(ctx, TP_ERR_MALFORMED, fn, "n = " + std::to_string(n) + " is not a power of two in [2, 2^28]");
  if (len != VK_HEAD + 64 * (size_t)n) return vk_fail(ctx, TP_ERR_MALFORMED, fn, "length does not match n");
  const size_t off_sig2 = OFF_SIG + 8 + 32 * (size_t)n;
  for (int s = 0; s < 2; s++) {
    uint64_t l;
    memcpy(&l, bytes + (s ? off_sig2 : OFF_SIG), 8);
    if (l != n) return vk_fail(ctx, TP_ERR_MALFORMED, fn, std::string(s ? "sigma_2" : "sigma_1") + " length is not n");
  }
  tp_vk* vk = new tp_vk();
  vk->ctx = ctx;
  vk->n = (size_t)n;
  while (((size_t)1 << vk->log_n) < vk->n) vk->log_n++;
  for (int i = 0; i < 3; i++) {
    uint64_t v[4];
    memcpy(v, bytes + OFF_K + 32 * i, 32);
    if (ge<4>(v, FR_PARAMS.mod)) {
      delete vk;
      return vk_fail(ctx, TP_ERR_MALFORMED, fn, "k[" + std::to_string(i) + "] not reduced modulo r");
    }
    vk->k[i] = HFr::to_mont(v);
  }
  uint8_t id_abi[TP_G1_BYTES];
  for (int i = 0; i < 9; i++) {
    if (!g1_record(bytes + OFF_G1 + 96 * i, check, i < 8 ? vk->com[i] : id_abi)) {
      delete vk;
      return vk_fail(ctx, TP_ERR_MALFORMED, fn, std::string("bad G1 point ") + kG1Names[i]);
    }
  }
  vk->identity = g1aff_decode(id_abi);
  if (vk->identity.inf) vk->identity = {HFq::zero(), HFq::one(), true};
  // the G2 points feed the pairings: they must be on the twist at every level, as tp_srs_deserialize requires
  G2Aff q, qs;
  if (!g2_from_wire(bytes + OFF_G2, check, &q) || !g2_on_curve(q)) {
    delete vk;
    return vk_fail(ctx, TP_ERR_MALFORMED, fn, "bad G2 point g2");
  }
  if (!g2_from_wire(bytes + OFF_G2S, check, &qs) || !g2_on_curve(qs)) {
    delete vk;
    return vk_fail(ctx, TP_ERR_MALFORMED, fn, "bad G2 point g2s");
  }
  vk->sp.g2 = q;
  vk->sp.g2s = qs;
  vk->sp.pg2 = g2_prepare(q);
  vk->sp.pg2s = g2_prepare(qs);
  // sigma_1 | sigma_2 through a 16-byte aligned staging buffer (the records sit at odd multiples of 8 in `bytes`),
  // and the nine G1 points' subgroup check (check 2) behind them
  int rc = alloc_sig(ctx, vk, fn);
  void* stage = nullptr;
  const size_t sig_bytes = 2 * vk->n * sizeof(Fr);
  if (rc == TP_OK && cudaMalloc(&stage, sig_bytes + 9 * sizeof(G1Affine) + 9) != cudaSuccess) {
    cudaGetLastError();
    stage = nullptr;
    rc = vk_fail(ctx, TP_ERR_CUDA, fn, "out of device memory");
  }
  size_t rejected = 0, first = 0;
  if (rc == TP_OK &&
      (cudaMemcpyAsync(stage, bytes + OFF_SIG + 8, sig_bytes / 2, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
       cudaMemcpyAsync((uint8_t*)stage + sig_bytes / 2, bytes + off_sig2 + 8, sig_bytes / 2, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess))
    rc = vk_fail(ctx, TP_ERR_CUDA, fn, "copy failed");
  if (rc == TP_OK) rc = fr_from_wire_dev(ctx, stage, 2 * vk->n, vk->sig, &rejected, &first);
  if (rc == TP_OK && rejected) {
    const bool second = first >= vk->n;
    rc = vk_fail(ctx, TP_ERR_MALFORMED, fn, std::to_string(rejected) + " sigma scalar(s) not reduced modulo r, first " +
                                                (second ? "sigma_2[" : "sigma_1[") + std::to_string(second ? first - vk->n : first) + "]");
  }
  if (rc == TP_OK && check >= 2) {
    std::vector<G1Affine> pts;
    std::vector<int> which;
    for (int i = 0; i < 9; i++) {
      const G1Aff p = i < 8 ? g1aff_decode(vk->com[i]) : vk->identity;
      if (p.inf) continue;   // the identity is in every subgroup (the device's record for it is not)
      pts.emplace_back();
      memcpy(&pts.back().x, p.x.v, 48);
      memcpy(&pts.back().y, p.y.v, 48);
      which.push_back(i);
    }
    uint8_t* dpts = (uint8_t*)stage + sig_bytes;
    uint8_t ok[9];
    if (!pts.empty()) {
      if (cudaMemcpyAsync(dpts, pts.data(), pts.size() * sizeof(G1Affine), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
        rc = vk_fail(ctx, TP_ERR_CUDA, fn, "copy failed");
      if (rc == TP_OK) rc = subgroup_flags_dev(ctx, (const G1Affine*)dpts, pts.size(), dpts + 9 * sizeof(G1Affine));
      if (rc == TP_OK && (cudaMemcpyAsync(ok, dpts + 9 * sizeof(G1Affine), pts.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                          cudaStreamSynchronize(ctx->stream) != cudaSuccess))
        rc = vk_fail(ctx, TP_ERR_CUDA, fn, "copy failed");
      for (size_t i = 0; rc == TP_OK && i < pts.size(); i++)
        if (!ok[i]) rc = vk_fail(ctx, TP_ERR_MALFORMED, fn, std::string("G1 point ") + kG1Names[which[i]] + " is not in the prime-order subgroup");
    }
  }
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = vk_fail(ctx, TP_ERR_CUDA, fn, "failed");
  if (stage) cudaFree(stage);
  if (rc != TP_OK) {
    free_key(vk);
    return rc;
  }
  *out = vk;
  return TP_OK;
}

}  // namespace

extern "C" {

int tp_vk_from_circuit(tp_ctx* ctx, tp_circuit* c, tp_vk** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !out) return fail(ctx, TP_ERR_INVALID_ARG, "vk_from_circuit: null argument");
  if (!ctx->children.empty()) {   // device group: every rank exports its own part (the commitment MSMs are sharded)
    if (c->parts.size() != ctx->children.size()) return fail(ctx, TP_ERR_INVALID_ARG, "vk_from_circuit: the circuit does not belong to this device group");
    return group_key(ctx, c->n, out, [&](tp_ctx* cc, int r, tp_vk** part) { return tp_vk_from_circuit(cc, c->parts[r], part); });
  }
  if (!c->srs->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "vk_from_circuit: the SRS has no G2 points (tp_srs_set_g2)");
  VerifierView view;
  TP_TRY(circuit_view(ctx, c, &view));
  tp_vk* vk = new tp_vk();
  vk->ctx = ctx;
  vk->n = c->n;
  vk->log_n = c->log_n;
  for (int i = 0; i < 3; i++) vk->k[i] = c->k[i];
  memcpy(vk->com, view.com, sizeof(vk->com));
  vk->identity = view.v.identity;
  vk->sp = *view.sp;
  int rc = alloc_sig(ctx, vk, "vk_from_circuit");
  for (int s = 0; s < 2 && rc == TP_OK; s++)
    if (cudaMemcpyAsync(vk->sig + s * vk->n, c->sig_coef[s], vk->n * sizeof(Fr), cudaMemcpyDeviceToDevice, ctx->stream) != cudaSuccess)
      rc = fail(ctx, TP_ERR_CUDA, "vk_from_circuit: copy failed");
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, TP_ERR_CUDA, "vk_from_circuit: copy failed");
  if (rc != TP_OK) {
    free_key(vk);
    return rc;
  }
  *out = vk;
  return TP_OK;
}

int tp_vk_destroy(tp_ctx* ctx, tp_vk* vk) {
  if (!vk) return TP_OK;
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!vk->parts.empty()) {
    group_run(ctx, [&](tp_ctx* cc, int r) { return tp_vk_destroy(cc, (size_t)r < vk->parts.size() ? vk->parts[r] : nullptr); });
    delete vk;
    return TP_OK;
  }
  cudaStreamSynchronize(ctx->stream);
  free_key(vk);
  return TP_OK;
}

int tp_vk_serialized_size(const tp_vk* vk, size_t* bytes) {
  if (!vk || !bytes) return TP_ERR_INVALID_ARG;
  *bytes = VK_HEAD + 64 * vk->n;
  return TP_OK;
}

int tp_vk_serialize(tp_ctx* ctx, const tp_vk* vk, uint8_t* out, size_t cap, size_t* written) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!vk || !out) return fail(ctx, TP_ERR_INVALID_ARG, "vk_serialize: null argument");
  if (vk->ctx != ctx) return fail(ctx, TP_ERR_INVALID_ARG, "vk_serialize: the key belongs to another context");
  if (!vk->parts.empty())   // device group: rank 0's part
    return group_run(ctx, [&](tp_ctx* c, int r) { return r == 0 ? tp_vk_serialize(c, vk->parts[0], out, cap, written) : TP_OK; });
  const size_t n = vk->n, need = VK_HEAD + 64 * n;
  if (written) *written = need;
  if (cap < need) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "vk_serialize: output buffer too small");
  memcpy(out, "TPVK", 4);
  const uint32_t version = 1;
  memcpy(out + 4, &version, 4);
  const uint64_t n64 = n;
  memcpy(out + OFF_N, &n64, 8);
  for (int i = 0; i < 3; i++) {
    HFr c = vk->k[i].from_mont();
    memcpy(out + OFF_K + 32 * i, c.v, 32);
  }
  for (int i = 0; i < 8; i++) serialize_g1_unchecked(vk->com[i], out + OFF_G1 + 96 * i);
  uint8_t id_abi[TP_G1_BYTES];
  memcpy(id_abi, vk->identity.x.v, 48);
  memcpy(id_abi + 48, vk->identity.y.v, 48);
  id_abi[96] = vk->identity.inf ? 1 : 0;
  serialize_g1_unchecked(id_abi, out + OFF_G1 + 96 * 8);
  g2_to_wire(vk->sp.g2, out + OFF_G2);
  g2_to_wire(vk->sp.g2s, out + OFF_G2S);
  const size_t off_sig2 = OFF_SIG + 8 + 32 * n;
  memcpy(out + OFF_SIG, &n64, 8);
  memcpy(out + off_sig2, &n64, 8);
  void* stage = nullptr;
  if (cudaMalloc(&stage, 2 * n * sizeof(Fr)) != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, TP_ERR_CUDA, "vk_serialize: out of device memory");
  }
  int rc = fr_to_wire_dev(ctx, vk->sig, 2 * n, stage);
  if (rc == TP_OK &&
      (cudaMemcpyAsync(out + OFF_SIG + 8, stage, 32 * n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
       cudaMemcpyAsync(out + off_sig2 + 8, (uint8_t*)stage + 32 * n, 32 * n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
       cudaStreamSynchronize(ctx->stream) != cudaSuccess))
    rc = fail(ctx, TP_ERR_CUDA, "vk_serialize: copy failed");
  cudaFree(stage);
  return rc;
}

int tp_vk_deserialize(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_vk** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!bytes || !out || check < 0 || check > 2) return fail(ctx, TP_ERR_INVALID_ARG, "vk_deserialize: null argument or check not in 0..2");
  if (!ctx->children.empty())   // device group: every rank decodes (and validates) its own part
    return group_key(ctx, 0, out, [&](tp_ctx* c, int, tp_vk** part) { return deserialize_one(c, bytes, len, check, part); });
  return deserialize_one(ctx, bytes, len, check, out);
}

int tp_vk_verify(tp_ctx* ctx, tp_vk* vk, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
                 size_t n_public, int* ok) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!vk || !proof || !ok || (n_public && !public_inputs)) return fail(ctx, TP_ERR_INVALID_ARG, "verify: null argument");
  if (vk->ctx != ctx) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify: the key belongs to another context");
  if (!vk->parts.empty()) {   // device group: every rank checks, the verdict is rank 0's (as tp_verify)
    std::vector<int> oks(ctx->children.size(), 0);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) { return tp_vk_verify(cc, vk->parts[r], proof, proof_len, public_inputs, n_public, &oks[r]); }));
    *ok = oks[0];
    return TP_OK;
  }
  return verify_single(ctx, vk->n, true, [&](VerifierView* view) { key_view(ctx, vk, view); return TP_OK; },
                       proof, proof_len, public_inputs, n_public, ok);
}

int tp_vk_verify_batch(tp_ctx* ctx, tp_vk* const* keys, size_t n_keys, const uint32_t* key_of, const uint8_t* proofs,
                       size_t count, const uint64_t* const* public_inputs, const size_t* n_public, int* all_ok,
                       int* each_ok) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!keys || !all_ok || (count && (!proofs || !n_public || !key_of)))
    return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: null argument");
  if (count > 65536) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: more than 65536 proofs");
  if (n_keys < 1 || n_keys > 4096) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: n_keys not in [1, 4096]");
  for (size_t j = 0; j < n_keys; j++) {
    if (!keys[j]) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: null key");
    if (keys[j]->ctx != ctx) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: a key belongs to another context");
  }
  // the bounds tp_verify enforces, for every proof against its own key
  for (size_t k = 0; k < count; k++) {
    if (key_of[k] >= n_keys) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: key index out of range");
    if (!n_public[k]) continue;
    if (!public_inputs || !public_inputs[k]) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: null public-input vector");
    if (n_public[k] > keys[key_of[k]]->n) return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: more public inputs than rows");
    for (size_t i = 0; i < n_public[k]; i++)
      if (ge<4>(public_inputs[k] + 4 * i, FR_PARAMS.mod))
        return fail(ctx, TP_ERR_INVALID_ARG, "vk_verify_batch: public input not reduced modulo r");
  }
  *all_ok = 0;
  if (count == 0) {
    *all_ok = 1;
    return TP_OK;
  }
  if (!ctx->children.empty()) {   // device group: every rank runs the batch, the MSMs are sharded by bucket
    const size_t world = ctx->children.size();
    std::vector<int> alls(world, 0), eaches(each_ok ? world * count : 0, 0);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) {
      std::vector<tp_vk*> parts(n_keys);
      for (size_t j = 0; j < n_keys; j++) parts[j] = keys[j]->parts[r];
      return tp_vk_verify_batch(cc, parts.data(), n_keys, key_of, proofs, count, public_inputs, n_public, &alls[r],
                                each_ok ? &eaches[(size_t)r * count] : nullptr);
    }));
    *all_ok = alls[0];
    if (each_ok) memcpy(each_ok, eaches.data(), count * sizeof(int));
    return TP_OK;
  }
  std::vector<VerifierView> views(n_keys);
  for (size_t j = 0; j < n_keys; j++) key_view(ctx, keys[j], &views[j]);
  return verify_batch_views(ctx, views.data(), n_keys, key_of, true, proofs, count, public_inputs, n_public, all_ok, each_ok);
}

}  // extern "C"
