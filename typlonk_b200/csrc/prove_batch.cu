// tp_prove_batch: many witnesses of one circuit in one call.  The stages of prove_resident (api.cu) run for a wave of
// W proofs at once -- one gate-check launch, one grand product, one numerator, one combine, one lincomb launch and two
// batched scans for the whole wave, the transforms through ntt_batch_dev and the commitments through msm_batch_dev in
// sets of 16 -- so a wave pays one host round trip per stage where a loop of tp_prove pays one per proof.  The host
// algebra between the stages is prove.h, the same code tp_prove runs, so proof k is byte-identical to tp_prove_inputs
// on the same inputs.
#include <algorithm>
#include <memory>

#include "common.cuh"
#include "prove.h"

using namespace tp;
using tph::HFr;

namespace {

// Proofs per wave: at most WAVE_CAP, and no more than fit WAVE_MEM_SHARE of the free device memory.  Going from 8 to 64
// proofs per wave saved another 13-17 % per proof at 2^10..2^16 on a B200 (DESIGN.md, "Batch proving"); at 64 a wave
// of 2^16 proofs holds 5.5 GiB, and larger waves were not measured.
constexpr size_t WAVE_CAP = 64;
constexpr double WAVE_MEM_SHARE = 0.5;
constexpr int MSM_SETS = 16;   // MSM_MAX_BATCH (msm.cu)

// The per-proof buffers of tp_circuit for one wave slot, offsets in Fr.  Every column is m = max(n, 8) long, so each
// starts 256-byte aligned; a slot is 44 m + 8 Fr (z_eval has n + 1 entries).
struct Layout {
  size_t m, adv_eval, pi_eval, adv_coef, pi_coef, z_coef, buf4, t, q, r, z_eval, stride;
  explicit Layout(size_t n) {
    m = n < 8 ? 8 : n;
    adv_eval = 0;          // 3 m, and pi_eval right behind: the four uploaded columns are one block
    pi_eval = 3 * m;
    adv_coef = 4 * m;      // 3 m
    pi_coef = 7 * m;
    z_coef = 8 * m;
    buf4 = 9 * m;          // 6 x 4 m: a4 b4 c4 z4 pi4 num4
    t = 33 * m;            // 3 m (t0 | t1 | t2, contiguous with stride n)
    q = 36 * m;            // 6 x m
    r = 42 * m;
    z_eval = 43 * m;       // n + 1
    stride = 44 * m + 8;
  }
};

struct BatchIn {
  const uint64_t* const* advice;
  const uint64_t* const* public_inputs;
  const size_t* n_public;
};

// Proves inputs first .. first + w - 1 in the circuit's wave buffers; writes their blocks (zeros where a proof fails)
// and statuses.
int prove_wave(tp_ctx* ctx, tp_circuit* c, const Layout& L, const BatchIn& in, size_t first, size_t w, uint8_t* proofs,
               int* status) {
  const size_t n = c->n, S = L.stride, m = L.m;
  const tp_srs* srs = c->srs;
  Fr* const E = c->wave;
  auto slot = [&](size_t j, size_t off) { return E + j * S + off; };

  // 1. upload, one gate-check launch for the wave, one read-back of the per-proof flags
  for (size_t j = 0; j < w; j++) {
    const size_t k = first + j;
    for (int i = 0; i < 3; i++)
      TP_CUDA_OK(ctx, cudaMemcpyAsync(slot(j, L.adv_eval + i * m), in.advice[3 * k + i], n * sizeof(Fr),
                                      cudaMemcpyHostToDevice, ctx->stream));
    const size_t np = in.n_public[k];
    if (np) TP_CUDA_OK(ctx, cudaMemcpyAsync(slot(j, L.pi_eval), in.public_inputs[k], np * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
    if (np < n) TP_CUDA_OK(ctx, cudaMemsetAsync(slot(j, L.pi_eval + np), 0, (n - np) * sizeof(Fr), ctx->stream));
  }
  const Fr* sel[5] = {c->sel_eval[0], c->sel_eval[1], c->sel_eval[2], c->sel_eval[3], c->sel_eval[4]};
  std::vector<unsigned> flags(w);
  {
    const Fr* adv[3] = {slot(0, L.adv_eval), slot(0, L.adv_eval + m), slot(0, L.adv_eval + 2 * m)};
    TP_TRY(gate_check_dev(ctx, sel, adv, slot(0, L.pi_eval), n, S, (int)w, flags.data()));
  }
  // the proofs that pass stay, moved down to slots 0 .. A - 1 in order
  std::vector<size_t> prf;   // slot -> input index
  std::vector<bool> pi_zero;
  for (size_t j = 0; j < w; j++) {
    if (flags[j] & 1u) {
      status[first + j] = TP_ERR_GATE_UNSATISFIED;
      continue;
    }
    const size_t a = prf.size();
    if (a != j)
      TP_CUDA_OK(ctx, cudaMemcpyAsync(slot(a, L.adv_eval), slot(j, L.adv_eval), 4 * m * sizeof(Fr), cudaMemcpyDeviceToDevice, ctx->stream));
    prf.push_back(first + j);
    pi_zero.push_back((flags[j] & 2u) == 0);
  }
  const size_t A = prf.size();
  if (A == 0) return TP_OK;

  // 2. interpolation (3 columns, 4 with non-zero public inputs) and the round-1 commitments
  std::vector<const Fr*> ins;
  std::vector<Fr*> outs;
  std::vector<const uint64_t*> cos;
  for (size_t a = 0; a < A; a++) {
    for (int i = 0; i < (pi_zero[a] ? 3 : 4); i++) {   // pi_eval follows the advice columns, pi_coef likewise
      ins.push_back(slot(a, L.adv_eval + i * m));
      outs.push_back(slot(a, L.adv_coef + i * m));
    }
    // a zero public-input polynomial: its coset evaluations are zeros, its transforms and evaluation are skipped
    if (pi_zero[a]) TP_CUDA_OK(ctx, cudaMemsetAsync(slot(a, L.buf4 + 4 * 4 * m), 0, 4 * n * sizeof(Fr), ctx->stream));
  }
  TP_TRY(ntt_batch_dev(ctx, ins.data(), outs.data(), nullptr, (int)ins.size(), c->log_n, true));
  struct Com {
    uint8_t v[4][TP_G1_BYTES];
    uint8_t* operator[](int i) { return v[i]; }
  };
  std::vector<Com> com(A);
  auto msm_sets = [&](const std::vector<const Fr*>& sets, uint8_t (*res)[TP_G1_BYTES]) -> int {
    for (size_t o = 0; o < sets.size(); o += MSM_SETS) {
      const int cnt = (int)std::min<size_t>(MSM_SETS, sets.size() - o);
      TP_TRY(msm_batch_dev(ctx, srs, sets.data() + o, cnt, n, res + o));
    }
    return TP_OK;
  };
  {
    std::vector<const Fr*> sets;
    for (size_t a = 0; a < A; a++)
      for (int i = 0; i < 3; i++) sets.push_back(slot(a, L.adv_coef + i * m));
    std::vector<uint8_t> res(sets.size() * TP_G1_BYTES);
    TP_TRY(msm_sets(sets, (uint8_t(*)[TP_G1_BYTES])res.data()));
    for (size_t a = 0; a < A; a++)
      for (int i = 0; i < 3; i++) memcpy(com[a][i], &res[(3 * a + i) * TP_G1_BYTES], TP_G1_BYTES);
  }
  std::vector<HFr> beta(A), gamma(A), alpha(A), zeta(A);
  for (size_t a = 0; a < A; a++) tph::challenges2({com[a][0], com[a][1], com[a][2]}, &beta[a], &gamma[a]);

  // 3. grand products (one pass, one read-back, one batch inversion), z interpolation and commitments
  std::unique_ptr<bool[]> zero_den(new bool[A]), closes(new bool[A]);
  {
    const Fr* v[3] = {slot(0, L.adv_eval), slot(0, L.adv_eval + m), slot(0, L.adv_eval + 2 * m)};
    const Fr* idp[3] = {c->id[0], c->id[1], c->id[2]};
    const Fr* sg[3] = {c->sig_eval[0], c->sig_eval[1], c->sig_eval[2]};
    TP_TRY(perm_grand_product_batch_dev(ctx, v, S, idp, sg, n, (int)A, beta.data(), gamma.data(), slot(0, L.z_eval), S,
                                        zero_den.get(), closes.get()));
  }
  ins.clear();
  outs.clear();
  for (size_t a = 0; a < A; a++) {
    ins.push_back(slot(a, L.z_eval));
    outs.push_back(slot(a, L.z_coef));
  }
  TP_TRY(ntt_batch_dev(ctx, ins.data(), outs.data(), nullptr, (int)A, c->log_n, true));
  {
    std::vector<const Fr*> sets(outs.begin(), outs.end());
    std::vector<uint8_t> res(A * TP_G1_BYTES);
    TP_TRY(msm_sets(sets, (uint8_t(*)[TP_G1_BYTES])res.data()));
    for (size_t a = 0; a < A; a++) memcpy(com[a][3], &res[a * TP_G1_BYTES], TP_G1_BYTES);
  }
  for (size_t a = 0; a < A; a++) tph::challenges2({com[a][0], com[a][1], com[a][2], com[a][3]}, &alpha[a], &zeta[a]);

  // 4. quotient: the coset transforms of every (proof, coset) pair, one numerator launch over them, the inverse coset
  // transforms and one combine launch.  Coset 0 is skipped where z closes, as tp_prove does.
  HFr gens[4];
  tpp::coset_gens(c->log_n, gens);
  std::unique_ptr<bool[]> skip0(new bool[A]);
  std::vector<unsigned> items;
  ins.clear();
  outs.clear();
  cos.clear();
  for (size_t a = 0; a < A; a++) {
    skip0[a] = closes[a] && !ctx->quotient_all_cosets;
    const size_t src[5] = {L.adv_coef, L.adv_coef + m, L.adv_coef + 2 * m, L.z_coef, L.pi_coef};
    for (unsigned k = skip0[a] ? 1u : 0u; k < 4; k++) {
      items.push_back((unsigned)a << 2 | k);
      for (int i = 0; i < (pi_zero[a] ? 4 : 5); i++) {
        ins.push_back(slot(a, src[i]));
        outs.push_back(slot(a, L.buf4 + (size_t)i * 4 * m + (size_t)k * n));
        cos.push_back(k == 0 ? nullptr : gens[k].v);
      }
    }
  }
  TP_TRY(ntt_batch_dev(ctx, ins.data(), outs.data(), cos.data(), (int)ins.size(), c->log_n, false));
  {
    QuotientArgs qa;
    for (int i = 0; i < 5; i++) qa.sel4[i] = c->sel4[i];
    for (int i = 0; i < 3; i++) {
      qa.sig4[i] = c->sig4[i];
      qa.adv4[i] = slot(0, L.buf4 + (size_t)i * 4 * m);
      qa.k[i] = c->k[i];
    }
    qa.z4 = slot(0, L.buf4 + 3 * 4 * m);
    qa.pi4 = slot(0, L.buf4 + 4 * 4 * m);
    qa.l0_4 = c->l0_4;
    TP_TRY(ntt_get_twiddles(ctx, c->log_n + 2, &qa.tw4));
    qa.out = slot(0, L.buf4 + 5 * 4 * m);
    qa.stride = S;
    qa.count = (int)A;
    qa.alpha = alpha.data();
    qa.beta = beta.data();
    qa.gamma = gamma.data();
    qa.n = n;
    TP_TRY(quotient_numerator_dev(ctx, qa, items.data(), (int)items.size()));
  }
  ins.clear();
  outs.clear();
  cos.clear();
  for (unsigned it : items) {
    const size_t a = it >> 2, k = it & 3u;
    ins.push_back(slot(a, L.buf4 + 5 * 4 * m + k * n));   // out of place into the dead coset slots of buf4[0]
    outs.push_back(slot(a, L.buf4 + k * n));
    cos.push_back(k == 0 ? nullptr : gens[k].v);
  }
  TP_TRY(ntt_batch_dev(ctx, ins.data(), outs.data(), cos.data(), (int)ins.size(), c->log_n, true));
  TP_TRY(quotient_combine_dev(ctx, slot(0, L.buf4), n, S, (int)A, skip0.get(), slot(0, L.t)));

  // 5. openings: the eight evaluations of every proof in one scan, then every r in one lincomb launch and one scan,
  // then the nine opening / quotient commitments of every proof
  const HFr omega = omega_for_log(c->log_n);
  std::vector<tpp::ProofEvals> pe(A);
  {
    std::vector<const Fr*> polys;
    std::vector<Fr*> quots;
    std::vector<Fr> points;
    for (size_t a = 0; a < A; a++) {
      const Fr* pp[8] = {slot(a, L.adv_coef), slot(a, L.adv_coef + m), slot(a, L.adv_coef + 2 * m), slot(a, L.z_coef),
                         slot(a, L.z_coef), c->sig_coef[0], c->sig_coef[1], slot(a, L.pi_coef)};
      for (int i = 0; i < (pi_zero[a] ? 7 : 8); i++) {
        polys.push_back(pp[i]);
        quots.push_back(i < 5 ? slot(a, L.q + i * m) : nullptr);
        points.push_back(to_dev(i == 4 ? zeta[a] * omega : zeta[a]));
      }
    }
    std::vector<HFr> ys(polys.size());
    TP_TRY(poly_open_batch_dev(ctx, polys.data(), n, points.data(), quots.data(), (int)polys.size(), ys.data()));
    size_t at = 0;
    for (size_t a = 0; a < A; a++) {
      for (int i = 0; i < 5; i++) pe[a].ev[i] = ys[at + i];
      pe[a].sig_bar[0] = ys[at + 5];
      pe[a].sig_bar[1] = ys[at + 6];
      pe[a].pi_bar = pi_zero[a] ? HFr::zero() : ys[at + 7];
      at += pi_zero[a] ? 7 : 8;
    }
  }
  {
    std::vector<HFr> s(A * (tpp::R_TERMS + 1));
    for (size_t a = 0; a < A; a++) tpp::lin_scalars(c->k, pe[a], alpha[a], beta[a], gamma[a], zeta[a], n, &s[a * (tpp::R_TERMS + 1)]);
    const LinTerm terms[tpp::R_TERMS] = {{c->sel_coef[0], 0}, {c->sel_coef[1], 0}, {c->sel_coef[2], 0},
                                         {c->sel_coef[3], 0}, {c->sel_coef[4], 0}, {slot(0, L.z_coef), S},
                                         {c->sig_coef[2], 0}, {slot(0, L.t), S}, {slot(0, L.t + n), S},
                                         {slot(0, L.t + 2 * n), S}};
    TP_TRY(lincomb_dev(ctx, terms, tpp::R_TERMS, s.data(), n, (int)A, slot(0, L.r), S));
  }
  std::vector<HFr> r_bar(A);
  {
    std::vector<const Fr*> polys;
    std::vector<Fr*> quots;
    std::vector<Fr> points;
    for (size_t a = 0; a < A; a++) {
      polys.push_back(slot(a, L.r));
      quots.push_back(slot(a, L.q + 5 * m));
      points.push_back(to_dev(zeta[a]));
    }
    TP_TRY(poly_open_batch_dev(ctx, polys.data(), n, points.data(), quots.data(), (int)A, r_bar.data()));
  }
  std::vector<uint8_t> res(9 * A * TP_G1_BYTES);
  {
    // per proof as tp_prove's batch: the six opening witnesses, then t0 t1 t2 (q[i][n-1] == 0, so length n is exact)
    std::vector<const Fr*> sets;
    for (size_t a = 0; a < A; a++) {
      for (int i = 0; i < 6; i++) sets.push_back(slot(a, L.q + i * m));
      for (int i = 0; i < 3; i++) sets.push_back(slot(a, L.t + i * n));
    }
    TP_TRY(msm_sets(sets, (uint8_t(*)[TP_G1_BYTES])res.data()));
  }
  for (size_t a = 0; a < A; a++) {
    const size_t k = prf[a];
    if (zero_den[a]) {
      status[k] = TP_ERR_ZERO_DENOMINATOR;
      continue;
    }
    const uint8_t(*outs9)[TP_G1_BYTES] = (const uint8_t(*)[TP_G1_BYTES])&res[9 * a * TP_G1_BYTES];
    uint8_t wit[6][TP_G1_BYTES], tcom[3][TP_G1_BYTES];
    for (int i = 0; i < 6; i++) memcpy(wit[i], outs9[i], TP_G1_BYTES);
    for (int i = 0; i < 3; i++) memcpy(tcom[i], outs9[6 + i], TP_G1_BYTES);
    tpp::write_proof(proofs + k * TP_PROOF_FIXED_BYTES, com[a].v, wit, tcom, pe[a].ev, zeta[a], r_bar[a]);
    status[k] = TP_OK;
  }
  return TP_OK;
}

// One rank (or a plain context): size the wave, grow the circuit's wave buffers, run the waves.
int prove_batch_one(tp_ctx* ctx, tp_circuit* c, size_t count, const BatchIn& in, uint8_t* proofs, int* status) {
  const Layout L(c->n);
  const size_t per = L.stride * sizeof(Fr);
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = 0;
  const double avail = (double)free_b + (double)c->wave_cap * (double)per;   // what the wave buffers hold is reusable
  size_t w = (size_t)(WAVE_MEM_SHARE * avail / (double)per);
  w = std::max<size_t>(1, std::min(w, std::min(WAVE_CAP, count)));
  if (comm_ready(ctx)) {
    // every rank runs the same MSMs (they are sharded by bucket): the group takes its smallest wave
    TP_TRY(ensure(ctx, ctx->misc[6], (size_t)ctx->world * sizeof(uint64_t)));
    uint64_t* all = (uint64_t*)ctx->misc[6].p;
    const uint64_t mine = w;
    TP_CUDA_OK(ctx, cudaMemcpyAsync(all + ctx->rank, &mine, sizeof(mine), cudaMemcpyHostToDevice, ctx->stream));
    TP_TRY(comm_allgather(ctx, all + ctx->rank, all, sizeof(uint64_t)));
    std::vector<uint64_t> ws(ctx->world);
    TP_CUDA_OK(ctx, cudaMemcpyAsync(ws.data(), all, ws.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint64_t v : ws) w = std::min<size_t>(w, (size_t)v);
  }
  if (w > c->wave_cap) {
    TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    if (c->wave) cudaFree(c->wave);
    c->wave = nullptr;
    c->wave_cap = 0;
    if (cudaMalloc(&c->wave, w * per) != cudaSuccess) {
      cudaGetLastError();
      c->wave = nullptr;
      return fail(ctx, TP_ERR_CUDA, "prove_batch: out of device memory for the wave buffers");
    }
    c->wave_cap = w;
  }
  ctx->stat_prove_batch_wave = (double)w;
  for (size_t first = 0; first < count; first += w)
    TP_TRY(prove_wave(ctx, c, L, in, first, std::min(w, count - first), proofs, status));
  return TP_OK;
}

}  // namespace

extern "C" {

int tp_prove_batch(tp_ctx* ctx, tp_circuit* c, size_t count, const uint64_t* const* advice,
                   const uint64_t* const* public_inputs, const size_t* n_public, uint8_t* proofs_out, size_t proofs_cap,
                   int* status) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c) return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: null argument");
  if (count > 65536) return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: more than 65536 proofs");
  if (count == 0) return TP_OK;
  if (!advice || !n_public || !proofs_out) return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: null argument");
  for (size_t k = 0; k < count; k++) {
    if (!advice[3 * k] || !advice[3 * k + 1] || !advice[3 * k + 2])
      return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: null witness column");
    if (n_public[k] > c->n) return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: more public inputs than rows");
    if (n_public[k] && (!public_inputs || !public_inputs[k]))
      return fail(ctx, TP_ERR_INVALID_ARG, "prove_batch: null public-input vector");
  }
  if (proofs_cap / TP_PROOF_FIXED_BYTES < count) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "prove_batch: proof buffer too small");
  const BatchIn in{advice, public_inputs, n_public};
  std::vector<int> st(count, TP_OK);
  memset(proofs_out, 0, count * TP_PROOF_FIXED_BYTES);
  if (!ctx->children.empty()) {   // device group: every rank runs the batch on its own part, rank 0's outputs go out
    const size_t world = ctx->children.size();
    std::vector<uint8_t> others((world - 1) * count * TP_PROOF_FIXED_BYTES, 0);
    std::vector<int> others_st((world - 1) * count, TP_OK);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) {
      if (r == 0) return prove_batch_one(cc, c->parts[0], count, in, proofs_out, st.data());
      return prove_batch_one(cc, c->parts[r], count, in, &others[(size_t)(r - 1) * count * TP_PROOF_FIXED_BYTES],
                             &others_st[(size_t)(r - 1) * count]);
    }));
    ctx->stat_prove_batch_wave = ctx->children[0]->stat_prove_batch_wave;
  } else {
    TP_TRY(prove_batch_one(ctx, c, count, in, proofs_out, st.data()));
  }
  if (status) {
    memcpy(status, st.data(), count * sizeof(int));
    return TP_OK;
  }
  for (size_t k = 0; k < count; k++)
    if (st[k] != TP_OK) {
      ctx->err = "prove_batch: proof " + std::to_string(k) + ": " +
                 (st[k] == TP_ERR_GATE_UNSATISFIED ? "gate constraints do not vanish on the domain"
                                                   : "permutation prove: zero denominator");
      return st[k];
    }
  return TP_OK;
}

}  // extern "C"
