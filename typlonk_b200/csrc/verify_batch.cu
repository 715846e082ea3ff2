// Batch verification: `count` proofs of one circuit (tp_verify_batch) or of several verification keys
// (tp_vk_verify_batch, verify_key.cu) checked with one batched MSM and one pairing product.
//
// Every KZG equation e(W, [tau]_2) = e(x W + C - y G, [1]_2) of every proof (six per proof, proof.rs:245-281 and the
// opening of the linearisation commitment, :441-503) is weighted by a scalar rho_{k,i} and summed:
//   e(L, [tau]_2) e(-R, [1]_2) = 1,  L = sum rho_{k,i} W_{k,i},  R = sum rho_{k,i} (x_{k,i} W_{k,i} + C_{k,i} - y_{k,i} G)
// with C_{k,5} = the linearisation commitment expanded into its bases (lin_scalars, verify.cu).  L and R are two MSMs
// over one base set (13 points per proof, the circuit commitments, srs[0] and G), run by msm_batch_dev over a temporary
// tp_srs.  The rho are drawn from a Blake2b-512 hash of everything the call receives, so they are a pure function of
// the inputs (the ranks of a device group agree) and a cheating prover cannot choose its proofs after them.  Proofs
// against keys of different SRSes are grouped by (G2, tau G2): each group has its own L and R, one pair of pairings each.
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
// A job is NP polynomials of length n (one verifying key's sigma_1, sigma_2) at K points; one launch runs every job.
// Block = ME_THREADS threads = Kp points x SB coefficient lanes (Kp * SB = ME_THREADS, Kp = 1 .. 128, per job).  The
// job's blocks are (point group y, coefficient range x); block (x, y) evaluates at points [y Kp, (y + 1) Kp) over the
// coefficients [x L, (x + 1) L).  Tiles of ME_TILE coefficients are staged in shared memory, high tile first; lane s
// takes the coefficients lo + s + j SB of the range and runs Horner in w = z^SB (one chain per polynomial), so that a
// tile is used by all Kp points of the block and small batches still fill the GPU.  The lane's sum is scaled by
// z^(lo + s), the lanes are summed in shared memory and the ranges by k_multi_eval_sum.
constexpr unsigned ME_THREADS = 128;
constexpr unsigned ME_TILE = 128;   // = ME_THREADS: one element of each polynomial per thread and tile

struct MultiEvalJob {
  const Fr* p[2];
  size_t n, range_len, ranges;
  size_t z0, K;        // the job's points: z[z0 .. z0 + K)
  size_t blk0;         // the job's blocks: [blk0, blk0 + ranges * groups), range-major within a point group
  size_t partial0;     // partial[partial0 + (q ranges + range) K + k]
  unsigned kp_log;     // Kp = 2^kp_log
};

struct MultiEvalArgs {
  const MultiEvalJob* jobs;   // device parameter block, ordered by blk0 and by z0
  unsigned njobs;
  const Fr* z;
  Fr* partial;
};

// the last job whose `field` is <= x (jobs ordered by that field)
template <size_t MultiEvalJob::*field>
__device__ __forceinline__ unsigned me_find(const MultiEvalJob* jobs, unsigned njobs, size_t x) {
  unsigned lo = 0, hi = njobs;
  while (hi - lo > 1) {
    const unsigned mid = (lo + hi) >> 1;
    if (jobs[mid].*field <= x) lo = mid; else hi = mid;
  }
  return lo;
}

template <int NP>
__global__ void __launch_bounds__(ME_THREADS) k_multi_eval(MultiEvalArgs a) {
  __shared__ Fr tile[NP][ME_TILE];
  const MultiEvalJob& J = a.jobs[me_find<&MultiEvalJob::blk0>(a.jobs, a.njobs, blockIdx.x)];
  const size_t local = blockIdx.x - J.blk0, ranges = J.ranges, K = J.K, n = J.n, range_len = J.range_len;
  const size_t range = local % ranges, group = local / ranges;
  const unsigned kp_log = J.kp_log;
  const unsigned tid = threadIdx.x;
  const unsigned kp = 1u << kp_log, sb = ME_THREADS >> kp_log;
  const unsigned pl = tid & (kp - 1), s = tid >> kp_log;
  const size_t pt = group * kp + pl;
  const bool live = pt < K;
  const size_t lo = range * range_len;
  const size_t hi = lo + range_len < n ? lo + range_len : n;
  const Fr* poly[NP];
#pragma unroll
  for (int q = 0; q < NP; q++) poly[q] = J.p[q];
  Fr* partial = a.partial + J.partial0;
  const Fr z = live ? fr_load(a.z + J.z0 + pt) : fr_zero();
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
    for (int q = 0; q < NP; q++) tile[q][tid] = k < hi ? fr_load(poly[q] + k) : fr_zero();
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
      fr_store(partial + ((size_t)q * ranges + range) * K + pt, sum);
    }
  }
}

// out[q Ktot + k] = sum over the ranges of k's job of its partial[q][range][k - z0]
__global__ void k_multi_eval_sum(MultiEvalArgs a, size_t Ktot, int np, Fr* out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)np * Ktot) return;
  const size_t q = i / Ktot, k = i % Ktot;
  const MultiEvalJob& J = a.jobs[me_find<&MultiEvalJob::z0>(a.jobs, a.njobs, k)];
  const size_t ranges = J.ranges, K = J.K;
  const Fr* partial = a.partial + J.partial0 + (k - J.z0);
  Fr sum = fr_zero();
  for (size_t r = 0; r < ranges; r++) sum = fr_add(sum, fr_load(partial + (q * ranges + r) * K));
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

// One job of multi_eval_dev: p[q](z_k) for q < np at the job's K points, which follow the earlier jobs' points in z.
struct EvalJob {
  const Fr* p[2];
  size_t n, K;
};

// Every job in one launch (z_dev, out_dev: device; z_dev holds the Ktot = sum K points job after job, out_dev gets
// np Ktot values, out_dev[q Ktot + k]).
int multi_eval_dev(tp_ctx* ctx, const EvalJob* jobs, size_t njobs, int np, const Fr* z_dev, Fr* out_dev) {
  ProfScope prof(ctx, TP_PHASE_SCAN);
  std::vector<MultiEvalJob> table;
  size_t blocks = 0, ktot = 0, partials = 0;
  for (size_t j = 0; j < njobs; j++) {
    const size_t n = jobs[j].n, K = jobs[j].K;
    if (!K) continue;   // a job owns at least one block and one point (me_find)
    unsigned kp_log = 0;
    while (kp_log < 7 && ((size_t)1 << kp_log) < K) kp_log++;
    const size_t kp = (size_t)1 << kp_log, sb = ME_THREADS / kp;
    const size_t groups = (K + kp - 1) / kp;
    // at least 64 coefficients per lane (the lane's z^(lo + s) is ~50 products), enough ranges for eight blocks per SM
    const size_t target = ((size_t)8 * ctx->sm_count + groups - 1) / groups;
    size_t range_len = std::max((size_t)64 * sb, (n + target - 1) / target);
    range_len = (range_len + ME_TILE - 1) / ME_TILE * ME_TILE;
    const size_t ranges = (n + range_len - 1) / range_len;
    table.emplace_back();
    MultiEvalJob& t = table.back();
    t.p[0] = jobs[j].p[0];
    t.p[1] = np > 1 ? jobs[j].p[1] : jobs[j].p[0];
    t.n = n;
    t.range_len = range_len;
    t.ranges = ranges;
    t.z0 = ktot;
    t.K = K;
    t.blk0 = blocks;
    t.partial0 = partials;
    t.kp_log = kp_log;
    blocks += ranges * groups;
    ktot += K;
    partials += (size_t)np * ranges * K;
  }
  if (!ktot) return TP_OK;
  if (blocks > 0x7fffffffu) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: evaluation grid too large");
  DevMem partial;
  TP_TRY(dev_alloc(ctx, partial, partials * sizeof(Fr)));
  MultiEvalArgs a;
  TP_TRY(params_upload(ctx, table.data(), table.size() * sizeof(MultiEvalJob), (const void**)&a.jobs));
  a.njobs = (unsigned)table.size();
  a.z = z_dev;
  a.partial = (Fr*)partial.p;
  if (np == 2)
    k_multi_eval<2><<<(unsigned)blocks, ME_THREADS, 0, ctx->stream>>>(a);
  else
    k_multi_eval<1><<<(unsigned)blocks, ME_THREADS, 0, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_multi_eval");
  const size_t outs = (size_t)np * ktot;
  k_multi_eval_sum<<<(unsigned)((outs + 255) / 256), 256, 0, ctx->stream>>>(a, ktot, np, out_dev);
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
const char kRhoKeysTag[] = "typlonk-verify-batch-keys-v1";

void g1aff_to_abi(const G1Aff& p, uint8_t out[TP_G1_BYTES]) {
  memcpy(out, p.x.v, 48);
  memcpy(out + 48, p.y.v, 48);
  out[96] = p.inf ? 1 : 0;
}

// The KZG equations of one proof as contributions to L and R (see the file comment).
constexpr int OWN_BASES = 13;    // wit[0..5] com[0..3] t[0..2]
constexpr int VIEW_BASES = 7;    // q_l q_r q_o q_m q_c sigma_3 identity of the proof's circuit / key
constexpr int GROUP_CHUNK = 8;   // SRS groups per msm_batch_dev call: two scalar vectors each (MSM_MAX_BATCH = 16)
struct Folded {
  HFr r_own[OWN_BASES];
  HFr l_own[6];
  HFr r_view[VIEW_BASES];
  HFr r_gen;
};

}  // namespace

int tpv::verify_batch_views(tp_ctx* ctx, const VerifierView* views, size_t n_views, const uint32_t* view_of,
                            bool keys_hash, const uint8_t* proofs, size_t count, const uint64_t* const* public_inputs,
                            const size_t* n_public, int* all_ok, int* each_ok) {
  auto vw = [view_of](size_t k) -> size_t { return view_of ? view_of[k] : 0; };
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

  // 3. sigma_1(zeta_k), sigma_2(zeta_k) in one launch over every view's coefficients (one job per view, its proofs'
  // points in a row); 4. PI(zeta_k)
  std::vector<VerifierValues> V(count);
  if (K) {
    std::vector<std::vector<size_t>> of_view(n_views);
    for (size_t k : alive) of_view[vw(k)].push_back(k);
    std::vector<size_t> order;
    std::vector<EvalJob> jobs;
    for (size_t j = 0; j < n_views; j++) {
      if (of_view[j].empty()) continue;
      jobs.push_back({{views[j].sig_coef[0], views[j].sig_coef[1]}, views[j].v.n, of_view[j].size()});
      order.insert(order.end(), of_view[j].begin(), of_view[j].end());
    }
    std::vector<Fr> zs(K);
    for (size_t i = 0; i < K; i++) zs[i] = to_dev(P[order[i]].point);
    DevMem dz, dy;
    TP_TRY(dev_alloc(ctx, dz, K * sizeof(Fr)));
    TP_TRY(dev_alloc(ctx, dy, 2 * K * sizeof(Fr)));
    TP_TRY(h2d_sync(ctx, dz.p, zs.data(), K * sizeof(Fr)));
    TP_TRY(multi_eval_dev(ctx, jobs.data(), jobs.size(), 2, (const Fr*)dz.p, (Fr*)dy.p));
    std::vector<Fr> ys(2 * K);
    TP_TRY(d2h_sync(ctx, ys.data(), dy.p, 2 * K * sizeof(Fr)));
    for (size_t i = 0; i < K; i++) {
      const size_t k = order[i];
      const VerifierView& view = views[vw(k)];
      V[k] = view.v;
      V[k].sigma_bar[0] = to_host(ys[i]);
      V[k].sigma_bar[1] = to_host(ys[K + i]);
      V[k].public_eval = HFr::zero();
      bool zero = true;
      for (size_t j = 0; j < 4 * n_public[k]; j++) zero &= public_inputs[k][j] == 0;
      if (zero) continue;   // PI = 0: every proof the reference can produce (SURVEY.md App. D.1)
      // tp_verify's route: pad, interpolate into the view's public-input buffers, evaluate at this proof's point
      const size_t n = view.v.n;
      Fr *eval, *coef;
      TP_TRY(view.pi_scratch(&eval, &coef));
      TP_CUDA_OK(ctx, cudaMemsetAsync(eval, 0, n * sizeof(Fr), ctx->stream));
      TP_CUDA_OK(ctx, cudaMemcpyAsync(eval, public_inputs[k], n_public[k] * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
      TP_TRY(ntt_dev(ctx, eval, coef, view.log_n, true, nullptr));
      const EvalJob pi = {{coef, coef}, n, 1};
      TP_TRY(multi_eval_dev(ctx, &pi, 1, 1, (const Fr*)dz.p + i, (Fr*)dy.p));
      Fr y;
      TP_TRY(d2h_sync(ctx, &y, dy.p, sizeof(Fr)));
      V[k].public_eval = to_host(y);
    }
  }

  // 5. rho_{k,i} = Fr::rand(StdRng::from_seed(Blake2b-512(tag | what binds the circuits | every proof)[0..32])).
  // One circuit (tp_verify_batch): n and its 8 commitments.  Keys: their count, then per key n, k, the nine G1 points
  // and the two G2 points (sigma_1, sigma_2 are bound by their commitments), and per proof its key index.
  std::vector<HFr> rho(count * 6);
  {
    Blake2b h;
    h.init();
    uint8_t ser[96];
    if (!keys_hash) {
      h.update((const uint8_t*)kRhoTag, sizeof(kRhoTag) - 1);
      uint64_t n64 = views[0].v.n;
      h.update((const uint8_t*)&n64, 8);
      for (int i = 0; i < 8; i++) {
        serialize_g1_unchecked(views[0].com[i], ser);
        h.update(ser, 96);
      }
    } else {
      h.update((const uint8_t*)kRhoKeysTag, sizeof(kRhoKeysTag) - 1);
      uint64_t nk = n_views;
      h.update((const uint8_t*)&nk, 8);
      for (size_t j = 0; j < n_views; j++) {
        const VerifierView& view = views[j];
        uint64_t n64 = view.v.n;
        h.update((const uint8_t*)&n64, 8);
        for (int i = 0; i < 3; i++) {
          HFr canon = view.v.k[i].from_mont();
          h.update((const uint8_t*)canon.v, 32);
        }
        for (int i = 0; i < 8; i++) {
          serialize_g1_unchecked(view.com[i], ser);
          h.update(ser, 96);
        }
        uint8_t id_abi[TP_G1_BYTES];
        g1aff_to_abi(view.v.identity, id_abi);
        serialize_g1_unchecked(id_abi, ser);
        h.update(ser, 96);
        uint8_t g2w[TP_WIRE_G2_BYTES];
        g2_to_wire(view.sp->g2, g2w);
        h.update(g2w, sizeof(g2w));
        g2_to_wire(view.sp->g2s, g2w);
        h.update(g2w, sizeof(g2w));
      }
    }
    for (size_t k = 0; k < count; k++) {   // the proof as tp_proof_encode writes it
      if (keys_hash) {
        uint32_t key = (uint32_t)vw(k);
        h.update((const uint8_t*)&key, 4);
      }
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
      const size_t k = alive[i];
      const HFr& z = P[k].point;
      if (z != HFr::one()) acc = acc * l0_denominator(V[k].n, z);
    }
    HFr inv = acc.inv();
    for (size_t i = K; i-- > 0;) {
      const size_t k = alive[i];
      const HFr& z = P[k].point;
      if (z == HFr::one()) continue;
      const HFr d = l0_denominator(V[k].n, z);
      l0[k] = (z.pow_u64(V[k].n) - HFr::one()) * inv * pre[i];
      inv = inv * d;
    }
  }
  std::vector<HFr> omega(n_views);
  for (size_t j = 0; j < n_views; j++) omega[j] = omega_for_log(views[j].log_n);
  std::vector<Folded> F(count);
  for (size_t k : alive) {
    const ParsedProof& p = P[k];
    const HFr* r = &rho[k * 6];
    HFr s[LIN_TERMS];
    lin_scalars(V[k], p, alpha[k], beta[k], gamma[k], l0[k], s);
    Folded& f = F[k];
    const HFr zeta = p.point, zeta_omega = zeta * omega[vw(k)];
    HFr gsum = HFr::zero();
    for (int i = 0; i < 6; i++) {
      f.l_own[i] = r[i];
      f.r_own[i] = r[i] * (i == 4 ? zeta_omega : zeta);
      if (i < 5) gsum = gsum + r[i] * p.ev[i];   // r is opened to 0, the value proof.rs:233 requires
    }
    for (int i = 0; i < 3; i++) f.r_own[6 + i] = r[i];
    f.r_own[9] = r[3] + r[4] + r[5] * s[LIN_Z];
    for (int i = 0; i < 3; i++) f.r_own[10 + i] = r[5] * s[LIN_T0 + i];
    for (int j = 0; j < 5; j++) f.r_view[j] = r[5] * s[LIN_QL + j];
    f.r_view[5] = r[5] * s[LIN_S3];
    f.r_view[6] = r[5] * s[LIN_ID];
    f.r_gen = HFr::zero() - gsum;
  }
  // the base set: every view's points, G, then 13 per proof; points at infinity are left out (xyzz_madd takes none)
  const G1Aff gen = {HFq::to_mont(G1_GEN_X), HFq::to_mont(G1_GEN_Y), false};
  std::vector<G1Affine> bases;
  std::vector<int> view_at(n_views * VIEW_BASES, -1), own_at(count * OWN_BASES, -1);
  int gen_at;
  {
    for (size_t j = 0; j < n_views; j++) {
      const VerifierValues& v = views[j].v;
      const G1Aff* vb[VIEW_BASES] = {&v.fixed[0], &v.fixed[1], &v.fixed[2], &v.fixed[3], &v.fixed[4], &v.sigma[2], &v.identity};
      for (int b = 0; b < VIEW_BASES; b++)
        if (!vb[b]->inf) {
          view_at[j * VIEW_BASES + b] = (int)bases.size();
          bases.emplace_back();
          g1_to_dev_record(*vb[b], &bases.back());
        }
    }
    gen_at = (int)bases.size();
    bases.emplace_back();
    g1_to_dev_record(gen, &bases.back());
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
  // SRS groups: views with the same (G2, tau G2) share one pair of MSMs and one pair of pairings
  std::vector<size_t> group_of(n_views), group_view;   // group_view[g]: the group's first view
  {
    std::vector<std::vector<uint8_t>> seen;
    for (size_t j = 0; j < n_views; j++) {
      std::vector<uint8_t> id(2 * TP_G2_BYTES);
      g2_encode(views[j].sp->g2, id.data());
      g2_encode(views[j].sp->g2s, id.data() + TP_G2_BYTES);
      size_t g = 0;
      while (g < seen.size() && seen[g] != id) g++;
      if (g == seen.size()) {
        seen.push_back(id);
        group_view.push_back(j);
      }
      group_of[j] = g;
    }
  }
  const size_t m = bases.size();
  const size_t chunk_vecs = 2 * std::min((size_t)GROUP_CHUNK, group_view.size());
  tp_srs* tmp = nullptr;
  DevMem dscal;
  if (K) {
    TP_TRY(srs_alloc(ctx, m, &tmp));
    int rc = h2d_sync(ctx, tmp->g1, bases.data(), m * sizeof(G1Affine));
    if (rc == TP_OK) rc = srs_build_levels_dev(ctx, tmp);
    if (rc == TP_OK) rc = dev_alloc(ctx, dscal, chunk_vecs * m * sizeof(Fr));
    if (rc != TP_OK) {
      tp_srs_destroy(ctx, tmp);
      return rc;
    }
  }
  std::unique_ptr<tp_srs, std::function<void(tp_srs*)>> tmp_guard(tmp, [ctx](tp_srs* s) { if (s) tp_srs_destroy(ctx, s); });
  // prod over the SRS groups g of e(L_g, tau_g G2) e(-R_g, G2_g) == 1 over the proofs of `set` (the scalars of every
  // other proof are zero); the groups with a proof in `set` go to the MSM GROUP_CHUNK at a time
  auto folded_check = [&](const std::vector<size_t>& set, bool* pass) -> int {
    std::vector<std::vector<size_t>> members(group_view.size());
    for (size_t k : set) members[group_of[vw(k)]].push_back(k);
    std::vector<size_t> active;
    for (size_t g = 0; g < members.size(); g++)
      if (!members[g].empty()) active.push_back(g);
    std::vector<G1Aff> ps;
    std::vector<const G2Prepared*> qs;
    std::vector<HFr> vacc(n_views * VIEW_BASES);
    for (size_t c0 = 0; c0 < active.size(); c0 += GROUP_CHUNK) {
      const size_t nc = std::min((size_t)GROUP_CHUNK, active.size() - c0);
      std::vector<Fr> sc(2 * nc * m);
      memset(sc.data(), 0, sc.size() * sizeof(Fr));
      for (size_t c = 0; c < nc; c++) {
        Fr* ls = sc.data() + 2 * c * m;
        Fr* rs = ls + m;
        HFr gacc = HFr::zero();
        std::vector<size_t> touched;
        for (size_t k : members[active[c0 + c]]) {
          const size_t j = vw(k);
          for (int b = 0; b < VIEW_BASES; b++) vacc[j * VIEW_BASES + b] = vacc[j * VIEW_BASES + b] + F[k].r_view[b];
          touched.push_back(j);
          gacc = gacc + F[k].r_gen;
          for (int b = 0; b < OWN_BASES; b++) {
            const int at = own_at[k * OWN_BASES + b];
            if (at < 0) continue;
            rs[at] = to_dev(F[k].r_own[b]);
            if (b < 6) ls[at] = to_dev(F[k].l_own[b]);
          }
        }
        for (size_t j : touched)
          for (int b = 0; b < VIEW_BASES; b++) {
            HFr& a = vacc[j * VIEW_BASES + b];
            const int at = view_at[j * VIEW_BASES + b];
            if (at >= 0 && !a.is_zero()) rs[at] = to_dev(a);
            a = HFr::zero();
          }
        rs[gen_at] = to_dev(gacc);
      }
      TP_TRY(h2d_sync(ctx, dscal.p, sc.data(), sc.size() * sizeof(Fr)));
      std::vector<const Fr*> vecs(2 * nc);
      for (size_t v = 0; v < 2 * nc; v++) vecs[v] = (const Fr*)dscal.p + v * m;
      std::vector<uint8_t> outs(2 * nc * TP_G1_BYTES);
      TP_TRY(msm_batch_dev(ctx, tmp, vecs.data(), (int)(2 * nc), m, (uint8_t(*)[TP_G1_BYTES])outs.data()));
      for (size_t c = 0; c < nc; c++) {
        const SrsPairing& sp = *views[group_view[active[c0 + c]]].sp;
        ps.push_back(g1aff_decode(&outs[2 * c * TP_G1_BYTES]));
        ps.push_back(g1_to_aff(g1_neg(g1_from_aff(g1aff_decode(&outs[(2 * c + 1) * TP_G1_BYTES])))));
        qs.push_back(&sp.pg2s);
        qs.push_back(&sp.pg2);
      }
    }
    *pass = pairing_product_is_one(ps.data(), qs.data(), (int)ps.size());
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
        for (size_t k : set) verdict[k] = verify_host(*views[vw(k)].sp, V[k], P[k]) ? 1 : 0;
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
  if (!c->srs->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "verify_batch: the SRS has no G2 points (tp_srs_set_g2)");
  VerifierView view;
  TP_TRY(circuit_view(ctx, c, &view));
  return verify_batch_views(ctx, &view, 1, nullptr, false, proofs, count, public_inputs, n_public, all_ok, each_ok);
}

}  // extern "C"
