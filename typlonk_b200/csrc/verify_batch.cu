// Batch verification: `count` proofs of one circuit checked with one MSM and one two-pair pairing product.
//
// Every KZG equation e(W, [tau]_2) = e(x W + C - y G, [1]_2) of every proof (six per proof, proof.rs:245-281 and the
// opening of the linearisation commitment, :441-503) is weighted by a scalar rho_{k,i} and summed:
//   e(L, [tau]_2) e(-R, [1]_2) = 1,  L = sum rho_{k,i} W_{k,i},  R = sum rho_{k,i} (x_{k,i} W_{k,i} + C_{k,i} - y_{k,i} G)
// with C_{k,5} = the linearisation commitment expanded into its bases (lin_scalars, verify.cu).  L and R are two MSMs
// over one base set (13 points per proof, the circuit commitments, srs[0] and G), run by msm_batch_dev over a temporary
// tp_srs.  The rho are drawn from a Blake2b-512 hash of everything the call receives, so they are a pure function of
// the inputs (the ranks of a device group agree) and a cheating prover cannot choose its proofs after them.
//
// Device work besides the MSM: [r]P = 0 for every proof point (one thread per point; random linear combinations are
// only sound on the r-torsion), and sigma_1, sigma_2 at every proof's challenge point (k_multi_eval: each coefficient
// is read from HBM once per group of up to 128 points).
#include "verify.h"
#include "transcript.h"

#include <algorithm>
#include <functional>
#include <memory>

using namespace tp;
using namespace tph;
using namespace tpv;

namespace {

// ---- multi-point evaluation ----------------------------------------------------------------------------------------
// Block = ME_THREADS threads = Kp points x SB coefficient lanes (Kp * SB = ME_THREADS, Kp = 1 .. 128).  Block (x, y)
// evaluates NP polynomials at points [y Kp, (y + 1) Kp) over the coefficients [x L, (x + 1) L).  Tiles of ME_TILE
// coefficients are staged in shared memory, high tile first; lane s takes the coefficients lo + s + j SB of the range
// and runs Horner in w = z^SB (one chain per polynomial), so that a tile is used by all Kp points of the block and
// small batches still fill the GPU.  The lane's sum is scaled by z^(lo + s), the lanes are summed in shared memory and
// the ranges by k_multi_eval_sum.
constexpr unsigned ME_THREADS = 128;
constexpr unsigned ME_TILE = 128;   // = ME_THREADS: one element of each polynomial per thread and tile

struct MultiEvalArgs {
  const Fr* p[2];
  const Fr* z;       // K points
  size_t n, K, range_len;
  unsigned kp_log;   // Kp = 2^kp_log
  Fr* partial;       // [NP][ranges][K]
};

template <int NP>
__global__ void __launch_bounds__(ME_THREADS) k_multi_eval(MultiEvalArgs a) {
  __shared__ Fr tile[NP][ME_TILE];
  const unsigned tid = threadIdx.x;
  const unsigned kp = 1u << a.kp_log, sb = ME_THREADS >> a.kp_log;
  const unsigned pl = tid & (kp - 1), s = tid >> a.kp_log;
  const size_t pt = (size_t)blockIdx.y * kp + pl;
  const bool live = pt < a.K;
  const size_t lo = (size_t)blockIdx.x * a.range_len;
  const size_t hi = lo + a.range_len < a.n ? lo + a.range_len : a.n;
  const Fr z = live ? fr_load(a.z + pt) : fr_zero();
  Fr w = z;
  for (unsigned i = sb; i > 1; i >>= 1) w = fr_sqr(w);
  Fr acc[NP];
#pragma unroll
  for (int q = 0; q < NP; q++) acc[q] = fr_zero();
  const size_t ntiles = (hi - lo + ME_TILE - 1) / ME_TILE;
  for (size_t t = ntiles; t-- > 0;) {
    const size_t k = lo + t * ME_TILE + tid;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NP; q++) tile[q][tid] = k < hi ? fr_load(a.p[q] + k) : fr_zero();
    __syncthreads();
    if (live)
      for (unsigned j = ME_TILE / sb; j-- > 0;) {
#pragma unroll
        for (int q = 0; q < NP; q++) acc[q] = fr_add(fr_mul(acc[q], w), tile[q][s + j * sb]);
      }
  }
  const Fr scale = fr_pow_u64(z, lo + s);
  __syncthreads();
#pragma unroll
  for (int q = 0; q < NP; q++) tile[q][tid] = fr_mul(acc[q], scale);
  __syncthreads();
  if (s == 0 && live) {
#pragma unroll
    for (int q = 0; q < NP; q++) {
      Fr sum = tile[q][pl];
      for (unsigned l = 1; l < sb; l++) sum = fr_add(sum, tile[q][l * kp + pl]);
      fr_store(a.partial + ((size_t)q * gridDim.x + blockIdx.x) * a.K + pt, sum);
    }
  }
}

// out[q K + k] = sum over the ranges of partial[q][range][k]
__global__ void k_multi_eval_sum(const Fr* partial, size_t ranges, size_t K, int np, Fr* out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)np * K) return;
  const size_t q = i / K, k = i % K;
  Fr sum = fr_zero();
  for (size_t r = 0; r < ranges; r++) sum = fr_add(sum, fr_load(partial + (q * ranges + r) * K + k));
  fr_store(out + i, sum);
}

// ok[i] = [r] pts[i] == identity (no point at infinity in pts)
__global__ void __launch_bounds__(128) k_subgroup_flags(const G1Affine* __restrict__ pts, size_t len, uint8_t* __restrict__ ok) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x)
    ok[i] = g1_in_subgroup(affine_load(pts + i)) ? 1 : 0;
}

}  // namespace

// An all-zero record (the device's infinity) gets 0: from (0, 0, 1, 1) every doubling gives the identity and every
// mixed addition (0, 0, 1, 1) again, and the ladder of the odd r ends with an addition.
int tp::subgroup_flags_dev(tp_ctx* ctx, const G1Affine* pts, size_t len, uint8_t* ok_dev) {
  if (len == 0) return TP_OK;
  const size_t blocks = std::min((len + 127) / 128, (size_t)ctx->sm_count * 16);
  k_subgroup_flags<<<(unsigned)blocks, 128, 0, ctx->stream>>>(pts, len, ok_dev);
  TP_LAUNCH(ctx, "k_subgroup_flags");
  return TP_OK;
}

namespace {

// device scratch of one call
struct DevMem {
  void* p = nullptr;
  ~DevMem() {
    if (p) cudaFree(p);
  }
};
int dev_alloc(tp_ctx* ctx, DevMem& m, size_t bytes) {
  if (cudaMalloc(&m.p, bytes ? bytes : 1) != cudaSuccess) {
    cudaGetLastError();
    m.p = nullptr;
    return fail(ctx, TP_ERR_CUDA, "verify_batch: out of device memory");
  }
  return TP_OK;
}

// p_q(z_k) for q < np, k < K (z_dev, out_dev: device; out_dev holds np K values)
int multi_eval_dev(tp_ctx* ctx, const Fr* const* polys, int np, size_t n, const Fr* z_dev, size_t K, Fr* out_dev) {
  ProfScope prof(ctx, TP_PHASE_SCAN);
  unsigned kp_log = 0;
  while (kp_log < 7 && ((size_t)1 << kp_log) < K) kp_log++;
  const size_t kp = (size_t)1 << kp_log, sb = ME_THREADS / kp;
  const size_t groups = (K + kp - 1) / kp;
  // at least 64 coefficients per lane (the lane's z^(lo + s) is ~50 products), enough ranges for eight blocks per SM
  const size_t target = ((size_t)8 * ctx->sm_count + groups - 1) / groups;
  size_t range_len = std::max((size_t)64 * sb, (n + target - 1) / target);
  range_len = (range_len + ME_TILE - 1) / ME_TILE * ME_TILE;
  const size_t ranges = (n + range_len - 1) / range_len;
  DevMem partial;
  TP_TRY(dev_alloc(ctx, partial, (size_t)np * ranges * K * sizeof(Fr)));
  MultiEvalArgs a;
  a.p[0] = polys[0];
  a.p[1] = np > 1 ? polys[1] : polys[0];
  a.z = z_dev;
  a.n = n;
  a.K = K;
  a.range_len = range_len;
  a.kp_log = kp_log;
  a.partial = (Fr*)partial.p;
  const dim3 grid((unsigned)ranges, (unsigned)groups);
  if (np == 2)
    k_multi_eval<2><<<grid, ME_THREADS, 0, ctx->stream>>>(a);
  else
    k_multi_eval<1><<<grid, ME_THREADS, 0, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_multi_eval");
  const size_t outs = (size_t)np * K;
  k_multi_eval_sum<<<(unsigned)((outs + 255) / 256), 256, 0, ctx->stream>>>(a.partial, ranges, K, np, out_dev);
  TP_LAUNCH(ctx, "k_multi_eval_sum");
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));   // before `partial` is freed
  return TP_OK;
}

int h2d_sync(tp_ctx* ctx, void* dst, const void* src, size_t bytes) {
  TP_CUDA_OK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}
int d2h_sync(tp_ctx* ctx, void* dst, const void* src, size_t bytes) {
  TP_CUDA_OK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}

void g1_to_dev_record(const G1Aff& p, G1Affine* out) {   // Montgomery x | y, the device SRS record
  memcpy(&out->x, p.x.v, 48);
  memcpy(&out->y, p.y.v, 48);
}

const char kRhoTag[] = "typlonk-verify-batch-v1";

// The KZG equations of one proof as contributions to L and R (see the file comment).
constexpr int OWN_BASES = 13;     // wit[0..5] com[0..3] t[0..2]
constexpr int SHARED_BASES = 8;   // q_l q_r q_o q_m q_c sigma_3 identity G
struct Folded {
  HFr r_own[OWN_BASES];
  HFr l_own[6];
  HFr r_shared[SHARED_BASES];
};

int verify_batch_one(tp_ctx* ctx, tp_circuit* c, const uint8_t* proofs, size_t count, const uint64_t* const* public_inputs,
                     const size_t* n_public, int* all_ok, int* each_ok) {
  if (!c->srs->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: the SRS has no G2 points (tp_srs_set_g2)");
  const SrsPairing& sp = *(const SrsPairing*)c->srs->pairing;
  const size_t n = c->n;
  std::vector<int> verdict(count, 0);
  // 1. parse, on the curve, challenge point, r(zeta) = 0: exact per-proof checks on the host
  std::vector<ParsedProof> P(count);
  std::vector<HFr> alpha(count), beta(count), gamma(count);
  std::vector<size_t> alive;
  for (size_t k = 0; k < count; k++) {
    ParsedProof& p = P[k];
    if (!parse_proof(proofs + k * TP_PROOF_FIXED_BYTES, &p) || !points_on_curve(p)) continue;
    HFr zeta;
    proof_challenges(p, &alpha[k], &beta[k], &gamma[k], &zeta);
    if (zeta != p.point || !p.r_eval.is_zero()) continue;
    alive.push_back(k);
  }
  VerifierValues base;
  TP_TRY(circuit_verifier_values(ctx, c, &base));

  // 2. [r]P = 0 for every finite point of the surviving proofs
  if (!alive.empty()) {
    std::vector<G1Affine> pts;
    std::vector<size_t> owner;
    pts.reserve(alive.size() * OWN_BASES);
    for (size_t k : alive) {
      const ParsedProof& p = P[k];
      const G1Aff* all[OWN_BASES] = {&p.wit[0], &p.wit[1], &p.wit[2], &p.wit[3], &p.wit[4], &p.wit[5], &p.com[0],
                                     &p.com[1], &p.com[2], &p.com[3], &p.t[0], &p.t[1], &p.t[2]};
      for (const G1Aff* g : all)
        if (!g->inf) {
          pts.emplace_back();
          g1_to_dev_record(*g, &pts.back());
          owner.push_back(k);
        }
    }
    if (!pts.empty()) {
      DevMem dpts, dok;
      TP_TRY(dev_alloc(ctx, dpts, pts.size() * sizeof(G1Affine)));
      TP_TRY(dev_alloc(ctx, dok, pts.size()));
      TP_CUDA_OK(ctx, cudaMemcpyAsync(dpts.p, pts.data(), pts.size() * sizeof(G1Affine), cudaMemcpyHostToDevice, ctx->stream));
      TP_TRY(subgroup_flags_dev(ctx, (const G1Affine*)dpts.p, pts.size(), (uint8_t*)dok.p));
      std::vector<uint8_t> ok(pts.size());
      TP_TRY(d2h_sync(ctx, ok.data(), dok.p, ok.size()));
      std::vector<char> bad(count, 0);
      for (size_t i = 0; i < ok.size(); i++)
        if (!ok[i]) bad[owner[i]] = 1;
      std::vector<size_t> keep;
      for (size_t k : alive)
        if (!bad[k]) keep.push_back(k);
      alive.swap(keep);
    }
  }
  const size_t K = alive.size();

  // 3. sigma_1(zeta_k), sigma_2(zeta_k) in one pass over the coefficients; 4. PI(zeta_k)
  std::vector<VerifierValues> V(count);
  if (K) {
    std::vector<Fr> zs(K);
    for (size_t i = 0; i < K; i++) zs[i] = to_dev(P[alive[i]].point);
    DevMem dz, dy;
    TP_TRY(dev_alloc(ctx, dz, K * sizeof(Fr)));
    TP_TRY(dev_alloc(ctx, dy, 2 * K * sizeof(Fr)));
    TP_TRY(h2d_sync(ctx, dz.p, zs.data(), K * sizeof(Fr)));
    const Fr* sig[2] = {c->sig_coef[0], c->sig_coef[1]};
    TP_TRY(multi_eval_dev(ctx, sig, 2, n, (const Fr*)dz.p, K, (Fr*)dy.p));
    std::vector<Fr> ys(2 * K);
    TP_TRY(d2h_sync(ctx, ys.data(), dy.p, 2 * K * sizeof(Fr)));
    for (size_t i = 0; i < K; i++) {
      const size_t k = alive[i];
      V[k] = base;
      V[k].sigma_bar[0] = to_host(ys[i]);
      V[k].sigma_bar[1] = to_host(ys[K + i]);
      V[k].public_eval = HFr::zero();
      bool zero = true;
      for (size_t j = 0; j < 4 * n_public[k]; j++) zero &= public_inputs[k][j] == 0;
      if (zero) continue;   // PI = 0: every proof the reference can produce (SURVEY.md App. D.1)
      // tp_verify's route: pad, interpolate into the prover's public-input buffers, evaluate at this proof's point
      TP_CUDA_OK(ctx, cudaMemsetAsync(c->pi_eval, 0, n * sizeof(Fr), ctx->stream));
      TP_CUDA_OK(ctx, cudaMemcpyAsync(c->pi_eval, public_inputs[k], n_public[k] * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
      c->pi_buffers_zero = false;
      TP_TRY(ntt_dev(ctx, c->pi_eval, c->pi_coef, c->log_n, true, nullptr));
      const Fr* pi[1] = {c->pi_coef};
      TP_TRY(multi_eval_dev(ctx, pi, 1, n, (const Fr*)dz.p + i, 1, (Fr*)dy.p));
      Fr y;
      TP_TRY(d2h_sync(ctx, &y, dy.p, sizeof(Fr)));
      V[k].public_eval = to_host(y);
    }
  }

  // 5. rho_{k,i} = Fr::rand(StdRng::from_seed(Blake2b-512(tag | n | 8 circuit commitments | every proof)[0..32]))
  std::vector<HFr> rho(count * 6);
  {
    Blake2b h;
    h.init();
    h.update((const uint8_t*)kRhoTag, sizeof(kRhoTag) - 1);
    uint64_t n64 = n;
    h.update((const uint8_t*)&n64, 8);
    for (int i = 0; i < 8; i++) {
      uint8_t ser[96];
      serialize_g1_unchecked(i < 5 ? c->fixed_com[i] : c->sigma_com[i - 5], ser);
      h.update(ser, 96);
    }
    for (size_t k = 0; k < count; k++) {   // the proof as tp_proof_encode writes it
      h.update(proofs + k * TP_PROOF_FIXED_BYTES, TP_PROOF_FIXED_BYTES);
      uint64_t np64 = n_public[k];
      h.update((const uint8_t*)&np64, 8);
      for (size_t j = 0; j < n_public[k]; j++) {
        HFr v;
        memcpy(v.v, public_inputs[k] + 4 * j, 32);
        HFr canon = v.from_mont();
        h.update((const uint8_t*)canon.v, 32);
      }
    }
    uint8_t digest[64];
    h.finalize(digest);
    StdRng rng = StdRng::from_seed(digest);
    for (auto& r : rho) r = fr_rand(rng);
  }

  // 6. fold: L_0(zeta_k) with one inversion for the whole batch, then each proof's scalars
  std::vector<HFr> l0(count, HFr::one());
  {
    std::vector<HFr> pre(K);
    HFr acc = HFr::one();
    for (size_t i = 0; i < K; i++) {
      pre[i] = acc;
      const HFr& z = P[alive[i]].point;
      if (z != HFr::one()) acc = acc * l0_denominator(n, z);
    }
    HFr inv = acc.inv();
    for (size_t i = K; i-- > 0;) {
      const HFr& z = P[alive[i]].point;
      if (z == HFr::one()) continue;
      const HFr d = l0_denominator(n, z);
      l0[alive[i]] = (z.pow_u64(n) - HFr::one()) * inv * pre[i];
      inv = inv * d;
    }
  }
  unsigned log_n = 0;
  while (((uint64_t)1 << log_n) < n) log_n++;
  const HFr omega = omega_for_log(log_n);
  std::vector<Folded> F(count);
  for (size_t k : alive) {
    const ParsedProof& p = P[k];
    const HFr* r = &rho[k * 6];
    HFr s[LIN_TERMS];
    lin_scalars(V[k], p, alpha[k], beta[k], gamma[k], l0[k], s);
    Folded& f = F[k];
    const HFr zeta = p.point, zeta_omega = zeta * omega;
    HFr gsum = HFr::zero();
    for (int i = 0; i < 6; i++) {
      f.l_own[i] = r[i];
      f.r_own[i] = r[i] * (i == 4 ? zeta_omega : zeta);
      if (i < 5) gsum = gsum + r[i] * p.ev[i];   // r is opened to 0, the value proof.rs:233 requires
    }
    for (int i = 0; i < 3; i++) f.r_own[6 + i] = r[i];
    f.r_own[9] = r[3] + r[4] + r[5] * s[LIN_Z];
    for (int i = 0; i < 3; i++) f.r_own[10 + i] = r[5] * s[LIN_T0 + i];
    for (int j = 0; j < 5; j++) f.r_shared[j] = r[5] * s[LIN_QL + j];
    f.r_shared[5] = r[5] * s[LIN_S3];
    f.r_shared[6] = r[5] * s[LIN_ID];
    f.r_shared[7] = HFr::zero() - gsum;
  }
  // the base set: shared points, then 13 per proof; points at infinity are left out (xyzz_madd takes none)
  const G1Aff gen = {HFq::to_mont(G1_GEN_X), HFq::to_mont(G1_GEN_Y), false};
  std::vector<G1Affine> bases;
  int shared_at[SHARED_BASES];
  std::vector<int> own_at(count * OWN_BASES, -1);
  {
    const G1Aff* shared[SHARED_BASES] = {&base.fixed[0], &base.fixed[1], &base.fixed[2], &base.fixed[3],
                                         &base.fixed[4], &base.sigma[2], &base.identity, &gen};
    for (int j = 0; j < SHARED_BASES; j++) {
      shared_at[j] = shared[j]->inf ? -1 : (int)bases.size();
      if (!shared[j]->inf) {
        bases.emplace_back();
        g1_to_dev_record(*shared[j], &bases.back());
      }
    }
    for (size_t k : alive) {
      const ParsedProof& p = P[k];
      const G1Aff* own[OWN_BASES] = {&p.wit[0], &p.wit[1], &p.wit[2], &p.wit[3], &p.wit[4], &p.wit[5], &p.com[0],
                                     &p.com[1], &p.com[2], &p.com[3], &p.t[0], &p.t[1], &p.t[2]};
      for (int b = 0; b < OWN_BASES; b++)
        if (!own[b]->inf) {
          own_at[k * OWN_BASES + b] = (int)bases.size();
          bases.emplace_back();
          g1_to_dev_record(*own[b], &bases.back());
        }
    }
  }
  const size_t m = bases.size();
  tp_srs* tmp = nullptr;
  DevMem dscal;
  if (K) {
    TP_TRY(srs_alloc(ctx, m, &tmp));
    int rc = h2d_sync(ctx, tmp->g1, bases.data(), m * sizeof(G1Affine));
    if (rc == TP_OK) rc = srs_build_levels_dev(ctx, tmp);
    if (rc == TP_OK) rc = dev_alloc(ctx, dscal, 2 * m * sizeof(Fr));
    if (rc != TP_OK) {
      tp_srs_destroy(ctx, tmp);
      return rc;
    }
  }
  std::unique_ptr<tp_srs, std::function<void(tp_srs*)>> tmp_guard(tmp, [ctx](tp_srs* s) { if (s) tp_srs_destroy(ctx, s); });
  // e(L, tau G2) e(-R, G2) == 1 over the proofs of `set` (the scalars of every other proof are zero)
  auto folded_check = [&](const std::vector<size_t>& set, bool* pass) -> int {
    std::vector<Fr> sc(2 * m);
    memset(sc.data(), 0, sc.size() * sizeof(Fr));
    Fr* ls = sc.data();
    Fr* rs = sc.data() + m;
    HFr shared[SHARED_BASES];
    for (auto& v : shared) v = HFr::zero();
    for (size_t k : set) {
      for (int j = 0; j < SHARED_BASES; j++) shared[j] = shared[j] + F[k].r_shared[j];
      for (int b = 0; b < OWN_BASES; b++) {
        const int at = own_at[k * OWN_BASES + b];
        if (at < 0) continue;
        rs[at] = to_dev(F[k].r_own[b]);
        if (b < 6) ls[at] = to_dev(F[k].l_own[b]);
      }
    }
    for (int j = 0; j < SHARED_BASES; j++)
      if (shared_at[j] >= 0) rs[shared_at[j]] = to_dev(shared[j]);
    TP_TRY(h2d_sync(ctx, dscal.p, sc.data(), sc.size() * sizeof(Fr)));
    const Fr* vecs[2] = {(const Fr*)dscal.p, (const Fr*)dscal.p + m};
    uint8_t outs[2][TP_G1_BYTES];
    TP_TRY(msm_batch_dev(ctx, tmp, vecs, 2, m, outs));
    G1Aff ps[2] = {g1aff_decode(outs[0]), g1_to_aff(g1_neg(g1_from_aff(g1aff_decode(outs[1]))))};
    const G2Prepared* qs[2] = {&sp.pg2s, &sp.pg2};
    *pass = pairing_product_is_one(ps, qs, 2);
    return TP_OK;
  };

  bool pass = false;
  if (K) TP_TRY(folded_check(alive, &pass));
  if (pass) {
    for (size_t k : alive) verdict[k] = 1;
  } else if (K && each_ok) {
    // 7. localise: halve the failing set and re-check each half; at most 8 proofs: tp_verify's host half, one by one
    std::function<int(const std::vector<size_t>&)> localise = [&](const std::vector<size_t>& set) -> int {
      if (set.size() <= 8) {
        for (size_t k : set) verdict[k] = verify_host(sp, V[k], P[k]) ? 1 : 0;
        return TP_OK;
      }
      const size_t half = set.size() / 2;
      const std::vector<size_t> parts[2] = {std::vector<size_t>(set.begin(), set.begin() + half),
                                            std::vector<size_t>(set.begin() + half, set.end())};
      for (const auto& part : parts) {
        bool ok = false;
        TP_TRY(folded_check(part, &ok));
        if (ok) {
          for (size_t k : part) verdict[k] = 1;
        } else {
          TP_TRY(localise(part));
        }
      }
      return TP_OK;
    };
    TP_TRY(localise(alive));
  }
  *all_ok = pass && K == count ? 1 : 0;
  if (each_ok)
    for (size_t k = 0; k < count; k++) each_ok[k] = verdict[k];
  return TP_OK;
}

}  // namespace

extern "C" {

int tp_verify_batch(tp_ctx* ctx, tp_circuit* c, const uint8_t* proofs, size_t count, const uint64_t* const* public_inputs,
                    const size_t* n_public, int* all_ok, int* each_ok) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !all_ok || (count && (!proofs || !n_public))) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: null argument");
  if (count > 65536) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: more than 65536 proofs");
  // the bounds tp_verify enforces, for every proof
  for (size_t k = 0; k < count; k++) {
    if (!n_public[k]) continue;
    if (!public_inputs || !public_inputs[k]) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: null public-input vector");
    if (n_public[k] > c->n) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: more public inputs than rows");
    for (size_t i = 0; i < n_public[k]; i++)
      if (ge<4>(public_inputs[k] + 4 * i, FR_PARAMS.mod))
        return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: public input not reduced modulo r");
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
      return tp_verify_batch(cc, c->parts[r], proofs, count, public_inputs, n_public, &alls[r],
                             each_ok ? &eaches[(size_t)r * count] : nullptr);
    }));
    *all_ok = alls[0];
    if (each_ok) memcpy(each_ok, eaches.data(), count * sizeof(int));
    return TP_OK;
  }
  return verify_batch_one(ctx, c, proofs, count, public_inputs, n_public, all_ok, each_ok);
}

}  // extern "C"
