// Internal shared declarations of libtyplonk_b200: context, device buffers, error plumbing,
// and the device-level entry points each .cu exports to the prover driver.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/typlonk_b200.h"
#include "ec.cuh"
#include "field.cuh"
#include "host_field.h"

namespace tp {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct LocalGroup;
struct MsmPipe;
struct NttTables {
  Fr* tw = nullptr;  // omega_N^i, i in [0, N/2]
};
struct CosetTable {
  unsigned log_n;
  uint64_t g[4];
  int scaled = 0;    // 1: every entry carries the factor n^-1 (inverse transforms)
  Fr* lo = nullptr;  // scale * g^i, i < 2^log_n
  Fr* hi = nullptr;  // unused (kept so that tp_ctx_destroy frees both)
};

}  // namespace tp

#define TP_PARAM_SLOTS 8

struct tp_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  int sm_count = 148;
  uint64_t launches = 0;
  // sharding (comm.cu): this context is rank `rank` of `world`; for world > 1 exactly one transport is set
  int rank = 0, world = 1;
  void* nccl = nullptr;                   // ncclComm_t owned by the library (tp_ctx_comm_init_rank / tp_ctx_create_multi)
  tp::LocalGroup* local = nullptr;        // ranks of one process without NCCL (several ranks on one device: tests)
  // device group (tp_ctx_create_multi): this context is only a front -- every entry point fans out to children[r]
  // (rank r, own device / stream / worker thread) and returns one result
  std::vector<tp_ctx*> children;
  void* workers = nullptr;
  // tunables (tp_ctx_set_option)
  unsigned msm_aff_rounds = 0;   // batch-affine rounds before the XYZZ accumulation (msm.cu 4a); 0 = off
  unsigned msm_affine_chains = 0;  // bucket accumulation in affine coordinates with per-thread batched inversion (msm.cu 4c)
  unsigned msm_reduce_l1 = 0;     // bucket reduction's running-sum level: 0 by size, 1 never, 2 whenever the set allows it
  unsigned quotient_all_cosets = 0;  // 1: evaluate the quotient numerator on all four cosets even when it is known to vanish on H
  unsigned msm_pipeline = 0;      // MSM batches as overlapped sub-batches on the pipe's own streams (msm.cu, "pipeline"):
                                  // 0 never (default: measured slower on 1 and on 8 GPUs), 1 on sharded contexts, 2 always
  unsigned msm_pipe_min_log = 15; // ... for inputs of at least 2^this points (tests lower it to reach the path with small circuits)
  unsigned ntt_radix_log = 2;     // butterfly stages per trip through registers: 3 (eight elements per thread) or 2 (four)
  unsigned msm_acc_staged = 0;    // 1: the accumulation stages the next table point in shared memory with cp.async
  unsigned msm_fq_lazy = 1;       // 1: the MSM's addition laws keep Fq values in [0, 2q) (ec.cuh FqOps<true>); 0: canonical
  // work counters (tp_ctx_get_stat)
  double stat_msm_entries = 0, stat_msm_calls = 0, stat_msm_c = 0, stat_msm_nwin = 0, stat_msm_levels = 0, stat_msm_chunk = 0;
  // profiling
  bool prof = false;
  double prof_ms[TP_PHASE_COUNT] = {0};
  uint64_t prof_launch[TP_PHASE_COUNT] = {0};
  struct Pending {
    int phase;
    cudaEvent_t a, b;
    uint64_t launches;
  };
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> event_pool;
  // caches
  std::map<unsigned, tp::NttTables> ntt_tables;
  std::vector<tp::CosetTable> coset_tables;
  // scratch
  tp::DevBuf ntt_scratch;
  // (the per-job buffers -- histogram, offsets, sorted list, buckets, partials, reduction levels -- live in the pipe's lanes)
  tp::DevBuf msm_scalars, msm_keys, msm_ranks, msm_blocksums, msm_winsums, msm_gather, msm_compact, msm_aff_pts, msm_sorted2,
      msm_aff_cnt, msm_aff_plan, msm_aff_rec;
  tp::MsmPipe* msm_pipe = nullptr;   // streams, lanes of scratch buffers and the queued sub-batches (msm.cu)
  tp::DevBuf scan_tmp[8];
  tp::DevBuf misc[16];
  tp::DevBuf flag;
  void* pinned = nullptr;  // small pinned staging area
  size_t pinned_cap = 0;
  void* fixed_base = nullptr;  // 32 x 255 affine multiples of G for SRS generation
  // tp_prove / tp_prove_inputs: the witness columns cross PCIe on their own stream, one event per column, so that
  // column k is interpolated while column k + 1 is still in flight (created on first use)
  // the prover's second compute stream (api.cu): challenge-independent coset NTTs run under the commitment MSMs
  cudaStream_t side_stream = nullptr;
  cudaEvent_t side_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[4] = {nullptr, nullptr, nullptr, nullptr};  // [0..2] column landed, [3] compute stream reached the upload
  // kernel parameter blocks (poly.cu params_upload): pinned staging, device copy and copy-done event per ring slot
  void* param_host[TP_PARAM_SLOTS] = {nullptr};
  size_t param_host_cap[TP_PARAM_SLOTS] = {0};
  tp::DevBuf param_dev[TP_PARAM_SLOTS];
  cudaEvent_t param_ev[TP_PARAM_SLOTS] = {nullptr};
  unsigned param_next = 0;
  // last tp_prove_batch: proofs per wave (tp_ctx_get_stat "prove_batch_wave")
  double stat_prove_batch_wave = 0;
};

struct tp_srs {
  // device, packed 96 B per point: `levels` copies of the SRS, g1[k * len + i] = 2^(c k) * [tau^i]G.
  // Level 0 is the SRS itself (what the ABI uploads / downloads); levels >= 1 are the fixed-base
  // window tables of the MSM (msm.cu), built once by srs_build_levels_dev.
  tp::G1Affine* g1 = nullptr;
  size_t len = 0;
  unsigned c = 0;       // MSM window bits the tables were built for
  unsigned levels = 1;
  void* pairing = nullptr;  // verify.cu: (G2, tau G2) with their Miller-loop line tables, and srs[0]
  std::vector<tp_srs*> parts;  // SRS of a device group: one full copy (with its table levels) per rank; nothing else is set
};

namespace tp {

#define TP_CUDA_OK(ctx, call)                                                                   \
  do {                                                                                          \
    cudaError_t e__ = (call);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                         \
      return TP_ERR_CUDA;                                                                       \
    }                                                                                           \
  } while (0)

#define TP_TRY(expr)             \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != TP_OK) return rc__; \
  } while (0)

inline int fail(tp_ctx* ctx, int code, const char* msg) {
  ctx->err = msg;
  return code;
}

// grow-only device buffer
inline int ensure(tp_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return TP_OK;
  if (b.p) {
    TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    TP_CUDA_OK(ctx, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes < 256 ? 256 : bytes;
  TP_CUDA_OK(ctx, cudaMalloc(&b.p, want));
  b.cap = want;
  return TP_OK;
}
inline void release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

inline int check_launch(tp_ctx* ctx, const char* what) {
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
    return TP_ERR_CUDA;
  }
  return TP_OK;
}
#define TP_LAUNCH(ctx, name) TP_TRY(tp::check_launch(ctx, name))

// Work queued while one of these is alive goes to `s` instead of the context's own stream.
struct StreamSwap {
  tp_ctx* c;
  cudaStream_t saved;
  StreamSwap(tp_ctx* ctx, cudaStream_t s) : c(ctx), saved(ctx->stream) { ctx->stream = s; }
  ~StreamSwap() { c->stream = saved; }
};

// ---- profiling scopes (CUDA events on the ctx stream) ---------------------------------
struct ProfScope {
  tp_ctx* ctx;
  int idx = -1;
  ProfScope(tp_ctx* c, int phase) : ctx(c) {
    if (!c->prof) return;
    tp_ctx::Pending p;
    p.phase = phase;
    auto get = [&]() {
      cudaEvent_t e;
      if (!c->event_pool.empty()) {
        e = c->event_pool.back();
        c->event_pool.pop_back();
      } else {
        cudaEventCreate(&e);
      }
      return e;
    };
    p.a = get();
    p.b = get();
    p.launches = c->launches;
    cudaEventRecord(p.a, c->stream);
    c->pending.push_back(p);
    idx = (int)c->pending.size() - 1;
  }
  ~ProfScope() {
    if (idx < 0) return;
    auto& p = ctx->pending[idx];
    cudaEventRecord(p.b, ctx->stream);
    p.launches = ctx->launches - p.launches;
  }
};

// ---- comm.cu: the two exchange steps of the sharded prover and the device-group plumbing ---------------
// every rank calls with the same sizes; ordered after the work already queued on ctx->stream
int comm_allgather(tp_ctx* ctx, const void* send_dev, void* recv_dev, size_t bytes_per_rank);
int comm_bcast(tp_ctx* ctx, void* dev_ptr, size_t bytes, int root);
int comm_group_begin(tp_ctx* ctx);   // broadcasts between begin and end run as one concurrent group (NCCL)
int comm_group_end(tp_ctx* ctx);
inline bool comm_ready(const tp_ctx* ctx) { return ctx->world > 1 && (ctx->nccl || ctx->local); }
void comm_release(tp_ctx* ctx);
// fn(children[r], r) on every worker thread of a group front at once; first non-zero status, error text copied up
int group_run(tp_ctx* group, const std::function<int(tp_ctx*, int)>& fn);
void group_destroy(tp_ctx* group);

// ---- device-level entry points (each implemented in its own .cu) -----------------------
// verify.cu
int srs_pairing_from_secret(tp_srs* srs, const tph::HFr& tau);
void srs_pairing_free(tp_srs* srs);
// ntt.cu
int ntt_dev(tp_ctx* ctx, const Fr* in, Fr* out, unsigned log_n, bool inverse, const uint64_t* coset);
int ntt_batch_dev(tp_ctx* ctx, const Fr* const* in, Fr* const* out, const uint64_t* const* coset, int count,
                  unsigned log_n, bool inverse);
int ntt_get_twiddles(tp_ctx* ctx, unsigned log_n, const Fr** tw);
tph::HFr omega_for_log(unsigned log_n);  // generator of the 2^log_n-th roots of unity (ark-poly Radix2EvaluationDomain)
int pow_table_dev(tp_ctx* ctx, Fr* out, const tph::HFr& base, size_t count);  // out[i] = base^i, i < count
// msm.cu : result as host Jacobian (this rank's shard only when sharded = false, else combined)
int msm_dev(tp_ctx* ctx, const tp_srs* srs, const Fr* scalars_dev, size_t len, uint8_t out[TP_G1_BYTES]);
// `batch` MSMs over the same bases in one pipeline (out[b] = sum_i scalars[b][i] * srs[i])
int msm_batch_dev(tp_ctx* ctx, const tp_srs* srs, const Fr* const* scalars_dev, int batch, size_t len,
                  uint8_t (*out)[TP_G1_BYTES]);
void encode_g1(const tph::HG1& p, uint8_t out[TP_G1_BYTES]);
// The same in two steps, so that the caller can queue other work in between: `submit` queues one sub-batch (its sort
// runs at once, under the accumulation of the sub-batch submitted before it), `finish` returns all results in
// submission order.  msm_pipe_overlaps: would a submit of this size run on the pipe's own streams?
int msm_pipe_submit(tp_ctx* ctx, const tp_srs* srs, const Fr* const* scalars_dev, int batch, size_t len);
int msm_pipe_finish(tp_ctx* ctx, uint8_t (*out)[TP_G1_BYTES], int count);
bool msm_pipe_overlaps(const tp_ctx* ctx, size_t len);
void msm_pipe_destroy(tp_ctx* ctx);
// poly.cu
// `bytes` of kernel parameters copied to the device in stream order; *dev stays valid for the launches queued next
int params_upload(tp_ctx* ctx, const void* src, size_t bytes, const void** dev);
// Several device entry points below work on `count` proofs at once: proof p's per-proof arrays sit at the given base
// pointer + p * stride (in Fr), circuit arrays are shared.  tp_prove calls them with count 1.
int perm_grand_product_dev(tp_ctx* ctx, const Fr* const values[3], const Fr* const id[3], const Fr* const sigma[3],
                           size_t n, const Fr& beta, const Fr& gamma, Fr* out /* n+1 */, bool* closes = nullptr);
// *closes (may be null): out[n] == 1, i.e. the copy constraints hold on the witness
// zero_den[p]: proof p has a zero denominator (its out is left undefined); closes[p] (may be null) as above
int perm_grand_product_batch_dev(tp_ctx* ctx, const Fr* const values[3], size_t vstride, const Fr* const id[3],
                                 const Fr* const sigma[3], size_t n, int count, const tph::HFr* beta,
                                 const tph::HFr* gamma, Fr* out, size_t ostride, bool* zero_den, bool* closes);
// q[k-1] = p[k] + z q[k]; writes q (len-1 coeffs, then a zero at [len-1]) and returns y = p(z)
int poly_open_dev(tp_ctx* ctx, const Fr* p, size_t len, const Fr& z, Fr* q_out /* len, may be null */, tph::HFr* y);
// any number of polynomials of the same length at once (own point each; q_out[b] may be null = evaluation only)
int poly_open_batch_dev(tp_ctx* ctx, const Fr* const* p, size_t len, const Fr* z, Fr* const* q_out, int batch, tph::HFr* y);
// flags[p] bit 0: the gate equation fails on some row of proof p; bit 1: some public input of proof p is non-zero
int gate_check_dev(tp_ctx* ctx, const Fr* const sel_evals[5], const Fr* const adv[3], const Fr* pi, size_t n,
                   size_t stride, int count, unsigned* flags);
struct QuotientArgs {   // every 4n-sized array is coset-major: slot k * n + i <-> omega_4n^(4i + k)
  const Fr* sel4[5];   // 4n evaluations
  const Fr* sig4[3];
  const Fr* l0_4;      // L0 on the 4n domain
  const Fr* tw4;       // omega_4n^i, i in [0, 2n]
  const Fr* adv4[3];   // per proof (+ p * stride)
  const Fr* z4;
  const Fr* pi4;
  Fr* out;             // 4n numerator evaluations
  size_t stride;
  int count;
  const tph::HFr* alpha;   // host, count each
  const tph::HFr* beta;
  const tph::HFr* gamma;
  tph::HFr k[3];
  size_t n;
};
// items[j] = proof << 2 | coset: one launch over every listed (proof, coset) pair
int quotient_numerator_dev(tp_ctx* ctx, const QuotientArgs& a, const unsigned* items, int nitems);
// t = floor(N / (X^n - 1)) (3n coefficients) from the four per-coset interpolants of N (coset-major, 4n)
// c0_is_zero[p]: coset 0 (H itself) of proof p was skipped because its numerator is known to vanish there
int quotient_combine_dev(tp_ctx* ctx, const Fr* c4, size_t n, size_t stride, int count, const bool* c0_is_zero,
                         Fr* t /* 3n */);
int l0_evals_4n_dev(tp_ctx* ctx, const Fr* tw4, size_t n, Fr* out /* 4n */);
struct LinTerm {
  const Fr* p;
  size_t stride;   // 0: shared by every proof
};
// out + p * ostride = scalars[p * (nterms + 1) + nterms] (at coefficient 0) + sum_t scalars[p * (nterms + 1) + t] * term t
int lincomb_dev(tp_ctx* ctx, const LinTerm* terms, int nterms, const tph::HFr* scalars, size_t n, int count, Fr* out,
                size_t ostride);
int sigma_tables_dev(tp_ctx* ctx, const uint64_t* perm_dev, size_t n, const Fr* tw, const Fr k[3], Fr* id[3],
                     Fr* sigma[3]);
int pad_copy_dev(tp_ctx* ctx, const Fr* in, size_t len, Fr* out, size_t out_len);
int rotate_copy_dev(tp_ctx* ctx, const Fr* in, size_t n, size_t shift, Fr* out);
void msm_choose_tables(size_t len, size_t table_len, size_t budget_bytes, unsigned world, unsigned* c_out, unsigned* levels_out);
// api.cu: device allocation of an SRS with the fixed-base table levels the MSM plan wants
int srs_alloc(tp_ctx* ctx, size_t len, tp_srs** out);
// api.cu: group front of an SRS, `make(rank context, &part)` on every rank (the rank is the context's `rank`)
int srs_group_new(tp_ctx* group, tp_srs** out, const std::function<int(tp_ctx*, tp_srs**)>& make);
// wire.cu: Montgomery SRS records <-> ark-serialize 0.3 uncompressed records, on the device
int g1_to_wire_dev(tp_ctx* ctx, const G1Affine* in, size_t len, void* out_dev);
int g1_from_wire_dev(tp_ctx* ctx, const void* in_dev, size_t len, int check, G1Affine* out, size_t* rejected,
                     size_t* first_rejected);
// wire.cu: Montgomery Fr <-> 32-byte canonical records (in_dev / out_dev 16-byte aligned); a record >= r is rejected
int fr_to_wire_dev(tp_ctx* ctx, const Fr* in, size_t len, void* out_dev);
int fr_from_wire_dev(tp_ctx* ctx, const void* in_dev, size_t len, Fr* out, size_t* rejected, size_t* first_rejected);
// srs.cu
int srs_generate_dev(tp_ctx* ctx, const tph::HFr& tau, size_t len, G1Affine* out);
int srs_build_levels_dev(tp_ctx* ctx, tp_srs* srs);
// out[i] = [s^i] in[i], i < len (level 0 only; the caller rebuilds the table levels)
int srs_contribute_dev(tp_ctx* ctx, const G1Affine* in, const tph::HFr& s, size_t len, G1Affine* out);
// verify_batch.cu: ok[i] = 1 iff [r] pts[i] is the identity (an all-zero record gets 0)
int subgroup_flags_dev(tp_ctx* ctx, const G1Affine* pts, size_t len, uint8_t* ok_dev);
// selftest.cu
int selftest_dev(tp_ctx* ctx, int* failures);
int measure_imad_dev(tp_ctx* ctx, double* imad, double* wide);

inline Fr to_dev(const tph::HFr& h) {
  Fr r;
  memcpy(r.v, h.v, 32);
  return r;
}
inline tph::HFr to_host(const Fr& d) {
  tph::HFr r;
  memcpy(r.v, d.v, 32);
  return r;
}

}  // namespace tp
