// Powers-of-tau ceremony over the device SRS: one contribution (tp_srs_contribute), the check that an SRS is the powers
// of one secret (tp_srs_verify) and the check of one contribution's link (tp_srs_update_check).  Additive API: the
// reference can only make an SRS from a secret one process holds (kzg/src/srs.rs:30-41).
//
// A contribution multiplies g1[i] by s^i on the device (k_srs_contribute, srs.cu), rebuilds the MSM's table levels
// and, on the host meanwhile, computes g2s' = [s] g2s and the pubkey [s]G2, which links the old SRS to the new one:
// e(g1'[1], G2) = e(g1[1], [s]G2).
//
// tp_srs_verify draws rho from the operating system after the SRS is fixed, computes M = sum_i rho^i g1[i] with one MSM
// over the SRS itself and accepts iff e(rho L, g2s) e(-D, G2) = 1 with L = M - rho^(n-1) g1[n-1], D = M - g1[0]
// (DESIGN.md, "Ceremony": sound because every g1[i] is checked to be in G1 first).
#include "verify.h"

#include <sys/random.h>

#include <array>
#include <cstdio>
#include <memory>

using namespace tp;
using namespace tph;
using tpv::SrsPairing;

namespace {

bool os_random_bytes(uint8_t* p, size_t n) {
  size_t got = 0;
  while (got < n) {
    ssize_t k = getrandom(p + got, n - got, 0);
    if (k <= 0) break;
    got += (size_t)k;
  }
  if (got < n) {
    std::FILE* f = std::fopen("/dev/urandom", "rb");
    if (f) {
      got += std::fread(p + got, 1, n - got, f);
      std::fclose(f);
    }
  }
  return got == n;
}

// uniform in Fr \ {0}: 255-bit draws below r, zero rejected (Montgomery form of the canonical draw)
int draw_nonzero_fr(tp_ctx* ctx, HFr* out) {
  for (;;) {
    uint64_t v[4];
    if (!os_random_bytes((uint8_t*)v, sizeof(v)))
      return fail(ctx, TP_ERR_INVALID_ARG, "srs_verify: no operating-system entropy source (getrandom, /dev/urandom)");
    v[3] &= ~(1ull << 63);
    if (ge<4>(v, FR_PARAMS.mod) || (v[0] | v[1] | v[2] | v[3]) == 0) continue;
    *out = HFr::to_mont(v);
    return TP_OK;
  }
}

bool g1_in_group(const G1Aff& p) { return g1_mul_u64limbs(g1_from_aff(p), FR_PARAMS.mod, 4).is_identity(); }
bool g2_in_group(const G2Aff& p) { return g2_mul(p, FR_PARAMS.mod, 4).inf; }
bool g2_is_generator(const G2Aff& p) {
  const G2Aff g = g2_generator();
  return !p.inf && p.x == g.x && p.y == g.y;
}

// a 97-byte ABI G1 record that is a canonical point of G1 other than the identity
bool g1_abi_in_group(const uint8_t in[TP_G1_BYTES], G1Aff* out) {
  *out = g1aff_decode(in);
  if (out->inf || ge<6>(out->x.v, FQ_PARAMS.mod) || ge<6>(out->y.v, FQ_PARAMS.mod)) return false;
  return g1aff_on_curve(*out) && g1_in_group(*out);
}
// a packed 96-byte device record (all zero = infinity)
G1Aff g1_from_record(const uint8_t in[96]) {
  G1Aff p;
  memcpy(p.x.v, in, 48);
  memcpy(p.y.v, in + 48, 48);
  p.inf = true;
  for (int i = 0; i < 96; i++) p.inf &= in[i] == 0;
  return p;
}

const tp_srs* first_part(const tp_srs* srs) { return srs->parts.empty() ? srs : srs->parts[0]; }

int contribute_one(tp_ctx* ctx, const tp_srs* srs, const HFr& s, tp_srs** out, uint8_t pubkey[TP_G2_BYTES]) {
  tp_srs* next = nullptr;
  TP_TRY(srs_alloc(ctx, srs->len, &next));
  int rc = srs_contribute_dev(ctx, srs->g1, s, srs->len, next->g1);
  if (rc == TP_OK) rc = srs_build_levels_dev(ctx, next);
  if (rc == TP_OK) {   // on the host while the device works
    const SrsPairing& sp = *(const SrsPairing*)srs->pairing;
    const HFr k = s.from_mont();
    uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
    g2_encode(sp.g2, g2);
    g2_encode(g2_mul(sp.g2s, k.v, 4), g2s);
    g2_encode(g2_mul(g2_generator(), k.v, 4), pubkey);
    rc = tp_srs_set_g2(next, g2, g2s);
  }
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, TP_ERR_CUDA, "srs_contribute: device work failed");
  if (rc != TP_OK) {
    tp_srs_destroy(ctx, next);
    return rc;
  }
  *out = next;
  return TP_OK;
}

// Every rank of a group runs this with the same rho: the MSM is sharded, so no rank may leave before it.
int verify_one(tp_ctx* ctx, const tp_srs* srs, const HFr& rho, int* ok) {
  const size_t n = srs->len;
  const SrsPairing& sp = *(const SrsPairing*)srs->pairing;
  *ok = 0;
  uint8_t* flags_dev = nullptr;
  TP_CUDA_OK(ctx, cudaMalloc(&flags_dev, n));
  std::unique_ptr<uint8_t, decltype(&cudaFree)> flags_guard(flags_dev, &cudaFree);
  TP_TRY(subgroup_flags_dev(ctx, srs->g1, n, flags_dev));
  TP_TRY(ensure(ctx, ctx->msm_scalars, n * sizeof(Fr)));
  TP_TRY(pow_table_dev(ctx, (Fr*)ctx->msm_scalars.p, rho, n));
  // the G2 half on the host while the device runs the ladders
  bool good = g2_is_generator(sp.g2) && !sp.g2s.inf && g2_on_curve(sp.g2s) && g2_in_group(sp.g2s);
  uint8_t m_abi[TP_G1_BYTES];
  TP_TRY(msm_dev(ctx, srs, (const Fr*)ctx->msm_scalars.p, n, m_abi));
  std::vector<uint8_t> flags(n);
  uint8_t first[96], last[96];
  TP_CUDA_OK(ctx, cudaMemcpyAsync(flags.data(), flags_dev, n, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaMemcpyAsync(first, srs->g1, 96, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaMemcpyAsync(last, srs->g1 + (n - 1), 96, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  for (size_t i = 0; i < n; i++) good &= flags[i] == 1;
  const HG1 gen = g1_from_affine(HFq::to_mont(G1_GEN_X), HFq::to_mont(G1_GEN_Y));
  G1Aff g0 = g1_from_record(first), gl = g1_from_record(last);
  good &= !g0.inf && g0.x == gen.x && g0.y == gen.y;
  if (!good) return TP_OK;
  // e(rho L, g2s) e(-D, G2) = 1:  L = M - rho^(n-1) g1[n-1] = sum_{i<n-1} rho^i g1[i],  D = M - g1[0]
  const HG1 m = g1_from_aff(g1aff_decode(m_abi));
  const HG1 l = g1_add(m, g1_neg(g1_mul_fr(g1_from_aff(gl), rho.pow_u64((uint64_t)(n - 1)))));
  const HG1 d = g1_add(m, g1_neg(g1_from_aff(g0)));
  const G1Aff ps[2] = {g1_to_aff(g1_mul_fr(l, rho)), g1_to_aff(g1_neg(d))};
  const G2Prepared* qs[2] = {&sp.pg2s, &sp.pg2};
  *ok = pairing_product_is_one(ps, qs, 2) ? 1 : 0;
  return TP_OK;
}

}  // namespace

extern "C" {

int tp_srs_contribute(tp_ctx* ctx, const tp_srs* srs, const uint64_t s[4], tp_srs** out, uint8_t pubkey[TP_G2_BYTES]) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!srs || !s || !out || !pubkey) return fail(ctx, TP_ERR_INVALID_ARG, "srs_contribute: null argument");
  if (ge<4>(s, FR_PARAMS.mod) || (s[0] | s[1] | s[2] | s[3]) == 0)
    return fail(ctx, TP_ERR_INVALID_ARG, "srs_contribute: the secret must be a non-zero element of Fr (Montgomery limbs below r)");
  if (!first_part(srs)->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "srs_contribute: the SRS has no G2 points (tp_srs_set_g2)");
  HFr k;
  memcpy(k.v, s, 32);
  if (!ctx->children.empty()) {   // every rank scales its own copy
    std::vector<std::array<uint8_t, TP_G2_BYTES>> keys(ctx->children.size());
    TP_TRY(srs_group_new(ctx, out, [&](tp_ctx* c, tp_srs** part) {
      return contribute_one(c, srs->parts[c->rank], k, part, keys[c->rank].data());
    }));
    memcpy(pubkey, keys[0].data(), TP_G2_BYTES);
    return TP_OK;
  }
  return contribute_one(ctx, srs, k, out, pubkey);
}

int tp_srs_verify(tp_ctx* ctx, const tp_srs* srs, int* ok) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!srs || !ok) return fail(ctx, TP_ERR_INVALID_ARG, "srs_verify: null argument");
  if (srs->len < 2) return fail(ctx, TP_ERR_INVALID_ARG, "srs_verify: fewer than two G1 points");
  if (!first_part(srs)->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "srs_verify: the SRS has no G2 points (tp_srs_set_g2)");
  *ok = 0;
  HFr rho;   // the verifier's private coin, drawn once the SRS is fixed
  TP_TRY(draw_nonzero_fr(ctx, &rho));
  if (!ctx->children.empty()) {   // one rho for every rank; the verdict is rank 0's
    std::vector<int> oks(ctx->children.size(), 0);
    TP_TRY(group_run(ctx, [&](tp_ctx* c, int r) { return verify_one(c, srs->parts[r], rho, &oks[r]); }));
    *ok = oks[0];
    return TP_OK;
  }
  return verify_one(ctx, srs, rho, ok);
}

int tp_srs_update_check(const uint8_t prev_tau_g1[TP_G1_BYTES], const uint8_t next_tau_g1[TP_G1_BYTES],
                        const uint8_t pubkey[TP_G2_BYTES], int* ok) {
  if (!prev_tau_g1 || !next_tau_g1 || !pubkey || !ok) return TP_ERR_INVALID_ARG;
  *ok = 0;
  G1Aff prev, next;
  if (!g1_abi_in_group(prev_tau_g1, &prev) || !g1_abi_in_group(next_tau_g1, &next)) return TP_OK;
  const G2Aff pk = g2_decode(pubkey);
  if (pk.inf || ge<6>(pk.x.a.v, FQ_PARAMS.mod) || ge<6>(pk.x.b.v, FQ_PARAMS.mod) || ge<6>(pk.y.a.v, FQ_PARAMS.mod) ||
      ge<6>(pk.y.b.v, FQ_PARAMS.mod) || !g2_on_curve(pk) || !g2_in_group(pk))
    return TP_OK;
  // e(next, G2) = e(prev, [s]G2)  <=>  e(next, G2) e(-prev, [s]G2) = 1
  const G2Prepared pg = g2_prepare(g2_generator()), ppk = g2_prepare(pk);
  const G1Aff ps[2] = {next, g1_to_aff(g1_neg(g1_from_aff(prev)))};
  const G2Prepared* qs[2] = {&pg, &ppk};
  *ok = pairing_product_is_one(ps, qs, 2) ? 1 : 0;
  return TP_OK;
}

}  // extern "C"
