// extern "C" surface of libtyplonk_b200 (include/typlonk_b200.h) and the device-resident
// prover driver that replaces plonk/src/proof.rs:96-194 (`prove`), :292-375
// (`quotient_polynomial`), :376-439 (`linearisation_poly`) and the setup numerics of
// plonk/src/builder.rs:70-88.  The host only sequences kernels, derives the Fiat-Shamir
// challenges (transcript.h) and does the O(1) scalar algebra between rounds.
#include "common.cuh"
#include "prove.h"

using namespace tp;
using tph::HFr;


static int dmalloc(tp_ctx* ctx, tp_circuit* c, Fr** p, size_t count) {
  void* v = nullptr;
  TP_CUDA_OK(ctx, cudaMalloc(&v, count * sizeof(Fr)));
  c->allocs.push_back(v);
  *p = (Fr*)v;
  return TP_OK;
}
static int h2d(tp_ctx* ctx, void* dst, const void* src, size_t bytes) {
  TP_CUDA_OK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return TP_OK;
}
static int d2h_sync(tp_ctx* ctx, void* dst, const void* src, size_t bytes) {
  TP_CUDA_OK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}
static unsigned log2_exact(size_t n) {
  unsigned l = 0;
  while (((size_t)1 << l) < n) l++;
  return l;
}

// ---- device groups (tp_ctx_create_multi, comm.cu) ----------------------------------------------------------------
// A group front holds no device state: every entry point below starts with a branch that runs the same entry point on
// every rank's own context from that rank's worker thread, and hands back rank 0's outputs (all ranks compute the same
// bytes).  Entry points without a collective inside run on rank 0 alone.
static inline bool is_group(const tp_ctx* ctx) { return ctx && !ctx->children.empty(); }
static int on_rank0(tp_ctx* g, const std::function<int(tp_ctx*)>& fn) {
  return group_run(g, [&](tp_ctx* c, int r) { return r == 0 ? fn(c) : TP_OK; });
}
#define TP_NO_GROUP(ctx, what)                                                                                          \
  do {                                                                                                                \
    if (is_group(ctx)) return fail(ctx, TP_ERR_INVALID_ARG, what ": device pointers belong to one device -- not available on a device group"); \
  } while (0)

static int mid_stream_priority() {
  int least = 0, greatest = 0;
  if (cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) return 0;
  return (least + greatest) / 2;   // numerically lower = more urgent; the range is [0, -5] on sm_100
}

extern "C" {

// ---- context ------------------------------------------------------------------------------
int tp_ctx_create(int device, void* stream, tp_ctx** out) {
  if (!out) return TP_ERR_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) return TP_ERR_NO_DEVICE;
  if (cudaSetDevice(device) != cudaSuccess) return TP_ERR_NO_DEVICE;
  tp_ctx* ctx = new tp_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  if (const char* v = getenv("TP_MSM_AFF_ROUNDS")) {
    long r = strtol(v, nullptr, 10);
    if (r >= 0 && r <= 8) ctx->msm_aff_rounds = (unsigned)r;
  }
  if (const char* v = getenv("TP_MSM_AFFINE")) ctx->msm_affine_chains = strtol(v, nullptr, 10) != 0 ? 1u : 0u;
  if (stream) {
    ctx->stream = (cudaStream_t)stream;
  } else {
    // middle priority: the MSM pipe puts its accumulation on a lowest-priority stream, so what the prover queues here
    // between two sub-batches (scans, transforms) gets SM slots ahead of the accumulation's pending blocks (msm.cu)
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, mid_stream_priority()) != cudaSuccess) {
      delete ctx;
      return TP_ERR_CUDA;
    }
    ctx->own_stream = true;
  }
  ctx->pinned_cap = 1 << 20;
  if (cudaMallocHost(&ctx->pinned, ctx->pinned_cap) != cudaSuccess) {
    delete ctx;
    return TP_ERR_CUDA;
  }
  *out = ctx;
  return TP_OK;
}

int tp_ctx_destroy(tp_ctx* ctx) {
  if (!ctx) return TP_OK;
  if (is_group(ctx)) {
    group_destroy(ctx);
    delete ctx;
    return TP_OK;
  }
  cudaSetDevice(ctx->device);
  comm_release(ctx);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->side_stream) {
    cudaStreamSynchronize(ctx->side_stream);
    cudaStreamDestroy(ctx->side_stream);
    for (auto& e : ctx->side_ev)
      if (e) cudaEventDestroy(e);
  }
  if (ctx->copy_stream) {
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamDestroy(ctx->copy_stream);
    for (auto& e : ctx->copy_ev)
      if (e) cudaEventDestroy(e);
  }
  for (auto& kv : ctx->ntt_tables) cudaFree(kv.second.tw);
  for (auto& c : ctx->coset_tables) {
    cudaFree(c.lo);
    cudaFree(c.hi);
  }
  msm_pipe_destroy(ctx);
  DevBuf* bufs[] = {&ctx->ntt_scratch, &ctx->msm_scalars, &ctx->msm_keys, &ctx->msm_ranks, &ctx->msm_blocksums,
                    &ctx->msm_winsums, &ctx->msm_gather, &ctx->msm_compact, &ctx->msm_aff_pts,
                    &ctx->msm_sorted2, &ctx->msm_aff_cnt, &ctx->msm_aff_plan, &ctx->msm_aff_rec, &ctx->flag};
  for (auto* b : bufs) release(*b);
  for (auto& b : ctx->scan_tmp) release(b);
  for (auto& b : ctx->misc) release(b);
  for (int s = 0; s < TP_PARAM_SLOTS; s++) {
    release(ctx->param_dev[s]);
    if (ctx->param_host[s]) cudaFreeHost(ctx->param_host[s]);
    if (ctx->param_ev[s]) cudaEventDestroy(ctx->param_ev[s]);
  }
  for (auto e : ctx->event_pool) cudaEventDestroy(e);
  for (auto& p : ctx->pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  if (ctx->fixed_base) cudaFree(ctx->fixed_base);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return TP_OK;
}

const char* tp_last_error(tp_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tp_sync(tp_ctx* ctx) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return group_run(ctx, [](tp_ctx* c, int) { return tp_sync(c); });
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}

int tp_ctx_set_option(tp_ctx* ctx, const char* name, long value) {
  if (!ctx || !name) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return group_run(ctx, [&](tp_ctx* c, int) { return tp_ctx_set_option(c, name, value); });
  if (strcmp(name, "msm_affine_rounds") == 0) {
    if (value < 0 || value > 8) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_affine_rounds must be 0..8");
    ctx->msm_aff_rounds = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_affine_chains") == 0) {
    if (value < 0 || value > 1) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_affine_chains must be 0 or 1");
    ctx->msm_affine_chains = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_reduce_l1") == 0) {
    if (value < 0 || value > 2) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_reduce_l1 must be 0, 1 or 2");
    ctx->msm_reduce_l1 = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_pipeline") == 0) {
    if (value < 0 || value > 2) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_pipeline must be 0, 1 or 2");
    ctx->msm_pipeline = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_fq_lazy") == 0) {
    if (value < 0 || value > 1) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_fq_lazy must be 0 or 1");
    ctx->msm_fq_lazy = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_pipe_min_log") == 0) {
    if (value < 0 || value > 27) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_pipe_min_log must be 0..27");
    ctx->msm_pipe_min_log = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "ntt_radix_log") == 0) {
    if (value < 2 || value > 3) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: ntt_radix_log must be 2 or 3");
    ctx->ntt_radix_log = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "msm_acc_staged") == 0) {
    if (value < 0 || value > 1) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: msm_acc_staged must be 0 or 1");
    ctx->msm_acc_staged = (unsigned)value;
    return TP_OK;
  }
  if (strcmp(name, "quotient_all_cosets") == 0) {
    if (value < 0 || value > 1) return fail(ctx, TP_ERR_INVALID_ARG, "set_option: quotient_all_cosets must be 0 or 1");
    ctx->quotient_all_cosets = (unsigned)value;
    return TP_OK;
  }
  return fail(ctx, TP_ERR_INVALID_ARG, "set_option: unknown option");
}

int tp_ctx_get_stat(tp_ctx* ctx, const char* name, double* out) {
  if (!ctx || !name || !out) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_ctx_get_stat(c, name, out); });
  const struct { const char* n; double v; } stats[] = {
      {"msm_entries", ctx->stat_msm_entries}, {"msm_calls", ctx->stat_msm_calls}, {"msm_window_bits", ctx->stat_msm_c},
      {"msm_windows", ctx->stat_msm_nwin},    {"msm_table_levels", ctx->stat_msm_levels}, {"msm_chunk", ctx->stat_msm_chunk},
      {"prove_batch_wave", ctx->stat_prove_batch_wave}};
  for (auto& st : stats)
    if (strcmp(name, st.n) == 0) {
      *out = st.v;
      return TP_OK;
    }
  return fail(ctx, TP_ERR_INVALID_ARG, "get_stat: unknown counter");
}

static int prof_collect(tp_ctx* ctx) {
  if (ctx->pending.empty()) return TP_OK;
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& p : ctx->pending) {
    float ms = 0;
    cudaEventElapsedTime(&ms, p.a, p.b);
    ctx->prof_ms[p.phase] += ms;
    ctx->prof_launch[p.phase] += p.launches;
    ctx->event_pool.push_back(p.a);
    ctx->event_pool.push_back(p.b);
  }
  ctx->pending.clear();
  return TP_OK;
}
int tp_prof_enable(tp_ctx* ctx, int on) {
  if (is_group(ctx)) return group_run(ctx, [&](tp_ctx* c, int) { return tp_prof_enable(c, on); });
  TP_TRY(prof_collect(ctx));
  ctx->prof = on != 0;
  return TP_OK;
}
int tp_prof_reset(tp_ctx* ctx) {
  if (is_group(ctx)) return group_run(ctx, [](tp_ctx* c, int) { return tp_prof_reset(c); });
  TP_TRY(prof_collect(ctx));
  for (int i = 0; i < TP_PHASE_COUNT; i++) {
    ctx->prof_ms[i] = 0;
    ctx->prof_launch[i] = 0;
  }
  ctx->stat_msm_entries = 0;
  ctx->stat_msm_calls = 0;
  return TP_OK;
}
int tp_prof_get(tp_ctx* ctx, double* ms, uint64_t* launches) {
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_prof_get(c, ms, launches); });   // rank 0's timers
  TP_TRY(prof_collect(ctx));
  for (int i = 0; i < TP_PHASE_COUNT; i++) {
    if (ms) ms[i] = ctx->prof_ms[i];
    if (launches) launches[i] = ctx->prof_launch[i];
  }
  return TP_OK;
}
int tp_launch_count(tp_ctx* ctx, uint64_t* out) {
  if (!ctx || !out) return TP_ERR_INVALID_ARG;
  *out = ctx->launches;
  for (tp_ctx* c : ctx->children) *out += c->launches;   // a group: kernels launched on all its devices
  return TP_OK;
}

// ---- SRS ------------------------------------------------------------------------------------
// Allocates the SRS with as many fixed-base table levels as the MSM plan wants and the device can
// spare (at most ~45 % of what is free; level 0 alone when nothing more fits).
extern "C++" {
namespace tp {
int srs_alloc(tp_ctx* ctx, size_t len, tp_srs** out) {
  tp_srs* s = new tp_srs();
  s->len = len;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = 0;
  size_t budget = (size_t)(0.45 * (double)free_b);
  // sharded by bucket, accumulation and reduction both shrink 1 / world: the window is the one a single GPU would pick
  // for the whole length (the rank count only enters through the fixed per-set overhead)
  for (int attempt = 0; attempt < 2; attempt++) {
    msm_choose_tables(len, len, attempt == 0 ? budget : 0, (unsigned)ctx->world, &s->c, &s->levels);
    cudaError_t e = cudaMalloc(&s->g1, (len ? len : 1) * (size_t)s->levels * sizeof(G1Affine));
    if (e == cudaSuccess) {
      *out = s;
      return TP_OK;
    }
    cudaGetLastError();
    s->g1 = nullptr;
  }
  delete s;
  return fail(ctx, TP_ERR_CUDA, "srs: out of device memory");
}

// group front of an SRS: `make(rank context, &part)` on every rank
int srs_group_new(tp_ctx* g, tp_srs** out, const std::function<int(tp_ctx*, tp_srs**)>& make) {
  tp_srs* front = new tp_srs();
  front->parts.assign(g->children.size(), nullptr);
  int rc = group_run(g, [&](tp_ctx* c, int r) { return make(c, &front->parts[r]); });
  if (rc != TP_OK) {
    group_run(g, [&](tp_ctx* c, int r) { return tp_srs_destroy(c, front->parts[r]); });
    delete front;
    return rc;
  }
  front->len = front->parts[0]->len;
  front->c = front->parts[0]->c;
  front->levels = front->parts[0]->levels;
  *out = front;
  return TP_OK;
}
}  // namespace tp
}  // extern "C++"

int tp_srs_from_secret(tp_ctx* ctx, const uint64_t tau[4], size_t gates, tp_srs** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!out || !tau) return fail(ctx, TP_ERR_INVALID_ARG, "srs_from_secret: null argument");
  if (is_group(ctx)) return srs_group_new(ctx, out, [&](tp_ctx* c, tp_srs** part) { return tp_srs_from_secret(c, tau, gates, part); });
  size_t len = gates + 3;
  tp_srs* s = nullptr;
  TP_TRY(srs_alloc(ctx, len, &s));
  HFr t;
  memcpy(t.v, tau, 32);
  int rc = srs_generate_dev(ctx, t, len, s->g1);
  if (rc == TP_OK) rc = srs_build_levels_dev(ctx, s);
  if (rc == TP_OK) rc = srs_pairing_from_secret(s, t);  // Srs::g2 (srs.rs:25-28), on the host while the device works
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, TP_ERR_CUDA, "srs: generation failed");
  if (rc != TP_OK) {
    srs_pairing_free(s);
    cudaFree(s->g1);
    delete s;
    return rc;
  }
  *out = s;
  return TP_OK;
}
int tp_srs_upload(tp_ctx* ctx, const uint8_t* g1_xy, size_t len, tp_srs** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!out || (!g1_xy && len)) return fail(ctx, TP_ERR_INVALID_ARG, "srs_upload: null argument");
  if (is_group(ctx)) return srs_group_new(ctx, out, [&](tp_ctx* c, tp_srs** part) { return tp_srs_upload(c, g1_xy, len, part); });
  tp_srs* s = nullptr;
  TP_TRY(srs_alloc(ctx, len, &s));
  int rc = h2d(ctx, s->g1, g1_xy, len * 96);
  if (rc == TP_OK) rc = srs_build_levels_dev(ctx, s);
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, TP_ERR_CUDA, "srs: upload failed");
  if (rc != TP_OK) {
    cudaFree(s->g1);
    delete s;
    return rc;
  }
  *out = s;
  return TP_OK;
}
int tp_srs_len(const tp_srs* srs, size_t* len) {
  if (!srs || !len) return TP_ERR_INVALID_ARG;
  *len = srs->len;
  return TP_OK;
}
int tp_srs_g1_download(tp_ctx* ctx, const tp_srs* srs, size_t offset, size_t count, uint8_t* out_xy) {
  if (!ctx || !srs) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_srs_g1_download(c, srs->parts[0], offset, count, out_xy); });
  if (offset + count > srs->len) return fail(ctx, TP_ERR_INVALID_ARG, "srs_download: range out of bounds");
  return d2h_sync(ctx, out_xy, srs->g1 + offset, count * 96);
}
int tp_srs_destroy(tp_ctx* ctx, tp_srs* srs) {
  if (!srs) return TP_OK;
  if (is_group(ctx)) {
    group_run(ctx, [&](tp_ctx* c, int r) { return tp_srs_destroy(c, (size_t)r < srs->parts.size() ? srs->parts[r] : nullptr); });
    delete srs;
    return TP_OK;
  }
  cudaStreamSynchronize(ctx->stream);
  cudaFree(srs->g1);
  srs_pairing_free(srs);
  delete srs;
  return TP_OK;
}

// ---- KZG ------------------------------------------------------------------------------------
int tp_commit_dev(tp_ctx* ctx, const tp_srs* srs, const void* coeffs_dev, size_t len, uint8_t out[TP_G1_BYTES]) {
  if (!ctx || !srs || !out) return TP_ERR_INVALID_ARG;
  TP_NO_GROUP(ctx, "commit_dev");
  return msm_dev(ctx, srs, (const Fr*)coeffs_dev, len, out);
}
int tp_commit(tp_ctx* ctx, const tp_srs* srs, const uint64_t* coeffs, size_t len, uint8_t out[TP_G1_BYTES]) {
  if (!ctx || !srs || !out || (len && !coeffs)) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) {
    std::vector<uint8_t> outs(ctx->children.size() * TP_G1_BYTES);
    TP_TRY(group_run(ctx, [&](tp_ctx* c, int r) { return tp_commit(c, srs->parts[r], coeffs, len, &outs[(size_t)r * TP_G1_BYTES]); }));
    memcpy(out, outs.data(), TP_G1_BYTES);
    return TP_OK;
  }
  if (len > srs->len) return fail(ctx, TP_ERR_SRS_TOO_SHORT, "commit: polynomial longer than the SRS");
  TP_TRY(ensure(ctx, ctx->msm_scalars, (len ? len : 1) * sizeof(Fr)));
  TP_TRY(h2d(ctx, ctx->msm_scalars.p, coeffs, len * sizeof(Fr)));
  return msm_dev(ctx, srs, (const Fr*)ctx->msm_scalars.p, len, out);
}
int tp_open(tp_ctx* ctx, const tp_srs* srs, const uint64_t* coeffs, size_t len, const uint64_t z[4],
            uint8_t w_out[TP_G1_BYTES], uint64_t y_out[4]) {
  if (!ctx || !srs || !z || !w_out || !y_out) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) {
    const size_t nr = ctx->children.size();
    std::vector<uint8_t> ws(nr * TP_G1_BYTES);
    std::vector<uint64_t> ys(nr * 4);
    TP_TRY(group_run(ctx, [&](tp_ctx* c, int r) {
      return tp_open(c, srs->parts[r], coeffs, len, z, &ws[(size_t)r * TP_G1_BYTES], &ys[(size_t)r * 4]);
    }));
    memcpy(w_out, ws.data(), TP_G1_BYTES);
    memcpy(y_out, ys.data(), 32);
    return TP_OK;
  }
  if (len == 0) return fail(ctx, TP_ERR_EMPTY_POLY, "open: empty polynomial");
  if (len > srs->len) return fail(ctx, TP_ERR_SRS_TOO_SHORT, "open: polynomial longer than the SRS");
  TP_TRY(ensure(ctx, ctx->msm_scalars, len * sizeof(Fr)));
  TP_TRY(ensure(ctx, ctx->misc[3], len * sizeof(Fr)));
  TP_TRY(h2d(ctx, ctx->misc[3].p, coeffs, len * sizeof(Fr)));
  Fr zd;
  memcpy(zd.v, z, 32);
  HFr y;
  TP_TRY(poly_open_dev(ctx, (const Fr*)ctx->misc[3].p, len, zd, (Fr*)ctx->msm_scalars.p, &y));
  memcpy(y_out, y.v, 32);
  return msm_dev(ctx, srs, (const Fr*)ctx->msm_scalars.p, len - 1, w_out);
}

// ---- NTT ------------------------------------------------------------------------------------
int tp_ntt_dev(tp_ctx* ctx, void* data_dev, unsigned log_n, int inverse, const uint64_t* coset) {
  if (!ctx || !data_dev) return TP_ERR_INVALID_ARG;
  TP_NO_GROUP(ctx, "ntt_dev");
  return ntt_dev(ctx, (const Fr*)data_dev, (Fr*)data_dev, log_n, inverse != 0, coset);
}
int tp_ntt(tp_ctx* ctx, uint64_t* data, unsigned log_n, int inverse, const uint64_t* coset) {
  if (!ctx || !data) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_ntt(c, data, log_n, inverse, coset); });   // one transform: one device
  if (log_n > 28) return fail(ctx, TP_ERR_INVALID_ARG, "ntt: log_n > 28");
  size_t n = (size_t)1 << log_n;
  TP_TRY(ensure(ctx, ctx->misc[3], n * sizeof(Fr)));
  TP_TRY(h2d(ctx, ctx->misc[3].p, data, n * sizeof(Fr)));
  TP_TRY(ntt_dev(ctx, (const Fr*)ctx->misc[3].p, (Fr*)ctx->misc[3].p, log_n, inverse != 0, coset));
  return d2h_sync(ctx, data, ctx->misc[3].p, n * sizeof(Fr));
}

// ---- permutation ------------------------------------------------------------------------------
int tp_perm_prove(tp_ctx* ctx, const uint64_t* const values[3], const uint64_t* const id[3],
                  const uint64_t* const sigma[3], size_t n, const uint64_t beta[4], const uint64_t gamma[4],
                  uint64_t* out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_perm_prove(c, values, id, sigma, n, beta, gamma, out); });
  if (n == 0) return fail(ctx, TP_ERR_INVALID_ARG, "perm_prove: n == 0");
  TP_TRY(ensure(ctx, ctx->misc[4], 9 * n * sizeof(Fr)));
  TP_TRY(ensure(ctx, ctx->misc[5], (n + 1) * sizeof(Fr)));
  Fr* base = (Fr*)ctx->misc[4].p;
  const Fr *v[3], *i_[3], *s[3];
  for (int k = 0; k < 3; k++) {
    TP_TRY(h2d(ctx, base + (size_t)k * n, values[k], n * sizeof(Fr)));
    TP_TRY(h2d(ctx, base + (size_t)(3 + k) * n, id[k], n * sizeof(Fr)));
    TP_TRY(h2d(ctx, base + (size_t)(6 + k) * n, sigma[k], n * sizeof(Fr)));
    v[k] = base + (size_t)k * n;
    i_[k] = base + (size_t)(3 + k) * n;
    s[k] = base + (size_t)(6 + k) * n;
  }
  Fr b, g;
  memcpy(b.v, beta, 32);
  memcpy(g.v, gamma, 32);
  TP_TRY(perm_grand_product_dev(ctx, v, i_, s, n, b, g, (Fr*)ctx->misc[5].p));
  return d2h_sync(ctx, out, ctx->misc[5].p, (n + 1) * sizeof(Fr));
}

// ---- circuit ------------------------------------------------------------------------------------
static int circuit_alloc(tp_ctx* ctx, tp_circuit* c) {
  size_t n = c->n;
  for (int i = 0; i < 5; i++) {
    TP_TRY(dmalloc(ctx, c, &c->sel_coef[i], n));
    TP_TRY(dmalloc(ctx, c, &c->sel_eval[i], n));
    TP_TRY(dmalloc(ctx, c, &c->sel4[i], 4 * n));
  }
  for (int i = 0; i < 3; i++) {
    TP_TRY(dmalloc(ctx, c, &c->id[i], n));
    TP_TRY(dmalloc(ctx, c, &c->sig_eval[i], n));
    TP_TRY(dmalloc(ctx, c, &c->sig_coef[i], n));
    TP_TRY(dmalloc(ctx, c, &c->sig4[i], 4 * n));
    TP_TRY(dmalloc(ctx, c, &c->adv_eval[i], n));
    TP_TRY(dmalloc(ctx, c, &c->adv_coef[i], n));
  }
  TP_TRY(dmalloc(ctx, c, &c->l0_4, 4 * n));
  TP_TRY(dmalloc(ctx, c, &c->pi_eval, n));
  TP_TRY(dmalloc(ctx, c, &c->pi_coef, n));
  TP_TRY(dmalloc(ctx, c, &c->z_eval, n + 1));
  TP_TRY(dmalloc(ctx, c, &c->z_coef, n));
  for (int i = 0; i < 6; i++) TP_TRY(dmalloc(ctx, c, &c->buf4[i], 4 * n));
  TP_TRY(dmalloc(ctx, c, &c->t, 3 * n));
  for (int i = 0; i < 6; i++) TP_TRY(dmalloc(ctx, c, &c->q[i], n));
  TP_TRY(dmalloc(ctx, c, &c->r, n));
  return TP_OK;
}

// coefficients (n) -> evaluations on coset k of the 4n domain, out4 coset-major (slot k * n + i)
static int to_coset(tp_ctx* ctx, tp_circuit* c, const Fr* coef, Fr* out4, unsigned k) {
  if (k == 0) return ntt_dev(ctx, coef, out4, c->log_n, false, nullptr);
  HFr g = omega_for_log(c->log_n + 2).pow_u64(k);
  return ntt_dev(ctx, coef, out4 + (size_t)k * c->n, c->log_n, false, g.v);
}
static int to_4n(tp_ctx* ctx, tp_circuit* c, const Fr* coef, Fr* out4) {
  for (unsigned k = 0; k < 4; k++) TP_TRY(to_coset(ctx, c, coef, out4, k));
  return TP_OK;
}

// derived data once sel_coef, id, sig_eval, k are in place
static int circuit_finish(tp_ctx* ctx, tp_circuit* c) {
  for (int i = 0; i < 5; i++) {
    TP_TRY(ntt_dev(ctx, c->sel_coef[i], c->sel_eval[i], c->log_n, false, nullptr));
    TP_TRY(to_4n(ctx, c, c->sel_coef[i], c->sel4[i]));
  }
  for (int i = 0; i < 3; i++) {
    TP_TRY(ntt_dev(ctx, c->sig_eval[i], c->sig_coef[i], c->log_n, true, nullptr));
    TP_TRY(to_4n(ctx, c, c->sig_coef[i], c->sig4[i]));
  }
  const Fr* tw4;
  TP_TRY(ntt_get_twiddles(ctx, c->log_n + 2, &tw4));
  TP_TRY(l0_evals_4n_dev(ctx, tw4, c->n, c->l0_4));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}

static int circuit_new(tp_ctx* ctx, const tp_srs* srs, size_t n, tp_circuit** out) {
  if (!out || !srs) return fail(ctx, TP_ERR_INVALID_ARG, "circuit: null argument");
  if (n < 2 || (n & (n - 1)) != 0 || n > ((size_t)1 << 26)) return fail(ctx, TP_ERR_INVALID_ARG, "circuit: n must be a power of two in [2, 2^26]");
  if (srs->len < n) return fail(ctx, TP_ERR_SRS_TOO_SHORT, "circuit: SRS shorter than the domain");
  tp_circuit* c = new tp_circuit();
  c->n = n;
  c->log_n = log2_exact(n);
  c->srs = srs;
  int rc = circuit_alloc(ctx, c);
  if (rc != TP_OK) {
    for (void* p : c->allocs) cudaFree(p);
    delete c;
    return rc;
  }
  *out = c;
  return TP_OK;
}

// group front of a circuit: `make(rank context, rank, &part)` on every rank
static int circuit_group_new(tp_ctx* g, const tp_srs* srs, size_t n, tp_circuit** out,
                             const std::function<int(tp_ctx*, int, tp_circuit**)>& make) {
  if (!out || !srs) return fail(g, TP_ERR_INVALID_ARG, "circuit: null argument");
  if (srs->parts.size() != g->children.size()) return fail(g, TP_ERR_INVALID_ARG, "circuit: the SRS does not belong to this device group");
  tp_circuit* front = new tp_circuit();
  front->n = n;
  front->log_n = log2_exact(n);
  front->srs = srs;
  front->parts.assign(g->children.size(), nullptr);
  int rc = group_run(g, [&](tp_ctx* c, int r) { return make(c, r, &front->parts[r]); });
  if (rc != TP_OK) {
    group_run(g, [&](tp_ctx* c, int r) { return tp_circuit_destroy(c, front->parts[r]); });
    delete front;
    return rc;
  }
  *out = front;
  return TP_OK;
}

int tp_circuit_destroy(tp_ctx* ctx, tp_circuit* c) {
  if (!c) return TP_OK;
  if (is_group(ctx)) {
    group_run(ctx, [&](tp_ctx* cc, int r) { return tp_circuit_destroy(cc, (size_t)r < c->parts.size() ? c->parts[r] : nullptr); });
    delete c;
    return TP_OK;
  }
  cudaStreamSynchronize(ctx->stream);
  for (void* p : c->allocs) cudaFree(p);
  if (c->wave) cudaFree(c->wave);
  delete c;
  return TP_OK;
}

int tp_circuit_load(tp_ctx* ctx, const tp_srs* srs, const uint64_t* const selectors[5], const uint64_t* const id[3],
                    const uint64_t* const sigma[3], const uint64_t cosets[3][4], size_t n, tp_circuit** out) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (is_group(ctx))
    return circuit_group_new(ctx, srs, n, out, [&](tp_ctx* c, int r, tp_circuit** part) {
      return tp_circuit_load(c, srs->parts[r], selectors, id, sigma, cosets, n, part);
    });
  tp_circuit* c = nullptr;
  TP_TRY(circuit_new(ctx, srs, n, &c));
  int rc = TP_OK;
  for (int i = 0; i < 5 && rc == TP_OK; i++) rc = h2d(ctx, c->sel_coef[i], selectors[i], n * sizeof(Fr));
  for (int i = 0; i < 3 && rc == TP_OK; i++) {
    rc = h2d(ctx, c->id[i], id[i], n * sizeof(Fr));
    if (rc == TP_OK) rc = h2d(ctx, c->sig_eval[i], sigma[i], n * sizeof(Fr));
    memcpy(c->k[i].v, cosets[i], 32);
  }
  if (rc == TP_OK) rc = circuit_finish(ctx, c);
  if (rc != TP_OK) {
    tp_circuit_destroy(ctx, c);
    return rc;
  }
  *out = c;
  return TP_OK;
}

int tp_circuit_compile(tp_ctx* ctx, const tp_srs* srs, const uint64_t* const selector_evals[5], const uint64_t* perm,
                       size_t n, tp_circuit** out, uint8_t fixed_commitments[5 * TP_G1_BYTES]) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!selector_evals || !perm || !out) return fail(ctx, TP_ERR_INVALID_ARG, "circuit_compile: null argument");
  if (is_group(ctx)) {
    std::vector<uint8_t> fixed(ctx->children.size() * 5 * TP_G1_BYTES);
    TP_TRY(circuit_group_new(ctx, srs, n, out, [&](tp_ctx* c, int r, tp_circuit** part) {
      return tp_circuit_compile(c, srs->parts[r], selector_evals, perm, n, part, &fixed[(size_t)r * 5 * TP_G1_BYTES]);
    }));
    if (fixed_commitments) memcpy(fixed_commitments, fixed.data(), 5 * TP_G1_BYTES);
    return TP_OK;
  }
  for (size_t i = 0; i < 3 * n; i++)   // k_sigma_tables splits an entry by / n and % n: out of range = a wrong sigma, silently
    if (perm[i] >= 3 * n) return fail(ctx, TP_ERR_INVALID_ARG, "circuit_compile: permutation index out of range");
  tp_circuit* c = nullptr;
  TP_TRY(circuit_new(ctx, srs, n, &c));
  int rc = TP_OK;
  // cosets (permutation/src/lib.rs:141-154): first three k >= 1 with k^n != 1
  {
    uint64_t kv = 1;
    for (int i = 0; i < 3; i++) {
      while (HFr::from_u64(kv).pow_u64((uint64_t)n) == HFr::one()) kv++;
      c->k[i] = HFr::from_u64(kv);
      kv++;
    }
  }
  // selectors: evaluations -> coefficients (builder.rs:84-86), then commit
  for (int i = 0; i < 5 && rc == TP_OK; i++) {
    rc = h2d(ctx, c->sel_eval[i], selector_evals[i], n * sizeof(Fr));
    if (rc == TP_OK) rc = ntt_dev(ctx, c->sel_eval[i], c->sel_coef[i], c->log_n, true, nullptr);
    if (rc == TP_OK) rc = msm_dev(ctx, srs, c->sel_coef[i], n, c->fixed_com[i]);
    if (rc == TP_OK && fixed_commitments) memcpy(fixed_commitments + i * TP_G1_BYTES, c->fixed_com[i], TP_G1_BYTES);
  }
  c->have_fixed_com = rc == TP_OK;
  // sigma / id tables (permutation/src/lib.rs:101-128)
  if (rc == TP_OK) {
    uint64_t* perm_dev = (uint64_t*)c->buf4[0];  // 3n u64 fits in a 4n Fr buffer
    rc = h2d(ctx, perm_dev, perm, 3 * n * sizeof(uint64_t));
    const Fr* tw;
    if (rc == TP_OK) rc = ntt_get_twiddles(ctx, c->log_n, &tw);
    Fr kd[3] = {to_dev(c->k[0]), to_dev(c->k[1]), to_dev(c->k[2])};
    if (rc == TP_OK) rc = sigma_tables_dev(ctx, perm_dev, n, tw, kd, c->id, c->sig_eval);
  }
  if (rc == TP_OK) rc = circuit_finish(ctx, c);
  if (rc != TP_OK) {
    tp_circuit_destroy(ctx, c);
    return rc;
  }
  *out = c;
  return TP_OK;
}

// Permutation::compile on its own (permutation/src/lib.rs:101-154): the (id, sigma) columns and the coset
// representatives of a flat permutation, computed by the kernel tp_circuit_compile uses.
int tp_permutation_compile(tp_ctx* ctx, const uint64_t* perm, size_t n, uint64_t* const id[3], uint64_t* const sigma[3],
                           uint64_t cosets[3][4]) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_permutation_compile(c, perm, n, id, sigma, cosets); });
  if (!perm || !id || !sigma || n == 0 || (n & (n - 1))) return fail(ctx, TP_ERR_INVALID_ARG, "permutation_compile: n must be a power of two");
  for (size_t i = 0; i < 3 * n; i++)
    if (perm[i] >= 3 * n) return fail(ctx, TP_ERR_INVALID_ARG, "permutation_compile: index out of range");
  const unsigned log_n = log2_exact(n);
  HFr k[3];
  uint64_t kv = 1;
  for (int i = 0; i < 3; i++) {
    while (HFr::from_u64(kv).pow_u64((uint64_t)n) == HFr::one()) kv++;
    k[i] = HFr::from_u64(kv);
    if (cosets) memcpy(cosets[i], k[i].v, 32);
    kv++;
  }
  TP_TRY(ensure(ctx, ctx->misc[0], 3 * n * sizeof(uint64_t)));
  TP_TRY(ensure(ctx, ctx->misc[1], 6 * n * sizeof(Fr)));
  TP_TRY(h2d(ctx, ctx->misc[0].p, perm, 3 * n * sizeof(uint64_t)));
  const Fr* tw;
  TP_TRY(ntt_get_twiddles(ctx, log_n, &tw));
  Fr kd[3] = {to_dev(k[0]), to_dev(k[1]), to_dev(k[2])};
  Fr* base = (Fr*)ctx->misc[1].p;
  Fr* idp[3] = {base, base + n, base + 2 * n};
  Fr* sgp[3] = {base + 3 * n, base + 4 * n, base + 5 * n};
  TP_TRY(sigma_tables_dev(ctx, (const uint64_t*)ctx->misc[0].p, n, tw, kd, idp, sgp));
  for (int i = 0; i < 3; i++) {
    TP_CUDA_OK(ctx, cudaMemcpyAsync(id[i], idp[i], n * sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA_OK(ctx, cudaMemcpyAsync(sigma[i], sgp[i], n * sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
  }
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}

int tp_circuit_sigma_commitments(tp_ctx* ctx, tp_circuit* c, uint8_t out[3 * TP_G1_BYTES]) {
  if (!ctx || !c || !out) return TP_ERR_INVALID_ARG;
  if (is_group(ctx)) {
    std::vector<uint8_t> outs(ctx->children.size() * 3 * TP_G1_BYTES);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) { return tp_circuit_sigma_commitments(cc, c->parts[r], &outs[(size_t)r * 3 * TP_G1_BYTES]); }));
    memcpy(out, outs.data(), 3 * TP_G1_BYTES);
    return TP_OK;
  }
  if (!c->have_sigma_com) {
    const Fr* sets[3] = {c->sig_coef[0], c->sig_coef[1], c->sig_coef[2]};
    TP_TRY(msm_batch_dev(ctx, c->srs, sets, 3, c->n, c->sigma_com));
    c->have_sigma_com = true;
  }
  memcpy(out, c->sigma_com, sizeof(c->sigma_com));
  return TP_OK;
}

// ---- prover -----------------------------------------------------------------------------------
// The prover's second stream: the forward coset NTTs of the quotient do not depend on any Fiat-Shamir challenge, so they
// are queued here as soon as their polynomial exists and run underneath the commitment MSMs of the main stream -- above
// all during the latency-bound tail of each MSM (bucket reduction, host round trip), when most SMs are idle.
static int side_stream_init(tp_ctx* ctx) {
  if (ctx->side_stream) return TP_OK;
  TP_CUDA_OK(ctx, cudaStreamCreateWithPriority(&ctx->side_stream, cudaStreamNonBlocking, mid_stream_priority()));
  for (auto& e : ctx->side_ev) TP_CUDA_OK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return TP_OK;
}
// rank that evaluates coset k of the 4n domain when cosets first..3 are to be done (first = 1: coset 0 skipped)
static int coset_owner(const tp_ctx* ctx, bool shard, unsigned first, unsigned k) {
  if (!shard) return ctx->rank;
  const unsigned ncos = 4u - first, j = k - first, world = (unsigned)ctx->world;
  return world < ncos ? (int)(j % world) : (int)(j * world / ncos);
}

// `col_ready` (may be null): three events on another stream, one per witness column, recorded when that column's
// upload has landed.  The prover then interpolates column k as soon as it is there -- while the next one is still
// crossing PCIe -- instead of waiting for all three and running the batched transform.
static int prove_resident(tp_ctx* ctx, tp_circuit* c, uint8_t* proof_out, const cudaEvent_t* col_ready = nullptr) {
  const size_t n = c->n;
  const tp_srs* srs = c->srs;
  // Quotient cosets of a, b, c on the side stream, under the round-1 MSMs.  Which cosets this rank owns depends on
  // whether coset 0 will be skipped (known only after the grand product): the honest case is assumed here and the
  // rest, if any, is done later.
  static const bool no_coset_shard = getenv("TP_NO_COSET_SHARD") && *getenv("TP_NO_COSET_SHARD") == '1';
  static const bool no_side_stream = getenv("TP_NO_SIDE_STREAM") && *getenv("TP_NO_SIDE_STREAM") == '1';
  const bool shard = comm_ready(ctx) && !no_coset_shard;
  HFr gens[4];
  tpp::coset_gens(c->log_n, gens);
  bool have[4][4] = {{false}};   // have[poly][coset]: evaluations of poly (a, b, c, z) on coset k are in buf4[poly]
  auto queue_cosets = [&](int poly_lo, int poly_hi, unsigned first) -> int {
    const Fr* src[4] = {c->adv_coef[0], c->adv_coef[1], c->adv_coef[2], c->z_coef};
    const Fr* ins[16];
    Fr* outs[16];
    const uint64_t* cos[16];
    int cnt = 0;
    for (unsigned k = first; k < 4; k++) {
      if (coset_owner(ctx, shard, first, k) != ctx->rank) continue;
      for (int i = poly_lo; i < poly_hi; i++) {
        if (have[i][k]) continue;
        have[i][k] = true;
        ins[cnt] = src[i];
        outs[cnt] = c->buf4[i] + (size_t)k * n;
        cos[cnt] = k == 0 ? nullptr : gens[k].v;
        cnt++;
      }
    }
    return ntt_batch_dev(ctx, ins, outs, cos, cnt, c->log_n, false);
  };
  const bool side = !no_side_stream;
  if (side) TP_TRY(side_stream_init(ctx));
  const unsigned first_guess = ctx->quotient_all_cosets ? 0u : 1u;
  // polynomials poly_lo .. poly_hi - 1 exist on the main stream: their quotient cosets go to the side stream
  auto side_cosets = [&](int poly_lo, int poly_hi, unsigned first, int ev) -> int {
    TP_CUDA_OK(ctx, cudaEventRecord(ctx->side_ev[ev], ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->side_stream, ctx->side_ev[ev], 0));
    {
      StreamSwap sw(ctx, ctx->side_stream);
      TP_TRY(queue_cosets(poly_lo, poly_hi, first));
    }
    TP_CUDA_OK(ctx, cudaEventRecord(ctx->side_ev[ev + 1], ctx->side_stream));
    return TP_OK;
  };
  if (col_ready) {
    // host buffers, one GPU: column k is interpolated as soon as its upload has landed, and its quotient cosets are
    // evaluated on the side stream while the next column is still crossing PCIe
    for (int k = 0; k < 3; k++) {
      TP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->stream, col_ready[k], 0));
      TP_TRY(ntt_dev(ctx, c->adv_eval[k], c->adv_coef[k], c->log_n, true, nullptr));
      if (side) TP_TRY(side_cosets(k, k + 1, first_guess, 0));
    }
  }
  // gate equation on every row (the reference asserts it via vanishes(line1), proof.rs:317-321) -- first, because it
  // needs nothing but the uploaded columns and also tells whether the public inputs are all zero.
  bool pi_zero = false;
  {
    unsigned flags = 0;
    const Fr* sel[5] = {c->sel_eval[0], c->sel_eval[1], c->sel_eval[2], c->sel_eval[3], c->sel_eval[4]};
    const Fr* adv[3] = {c->adv_eval[0], c->adv_eval[1], c->adv_eval[2]};
    TP_TRY(gate_check_dev(ctx, sel, adv, c->pi_eval, n, 0, 1, &flags));
    pi_zero = (flags & 2u) == 0;
    if (flags & 1u) return fail(ctx, TP_ERR_GATE_UNSATISFIED, "prove: gate constraints do not vanish on the domain");
  }
  // A zero public-input vector (the only kind the reference's prover accepts, SURVEY.md App. D.1) interpolates to the
  // zero polynomial: its inverse NTT, its four coset NTTs and its evaluation are skipped and the buffers just hold zeros.
  if (pi_zero && !c->pi_buffers_zero) {
    TP_CUDA_OK(ctx, cudaMemsetAsync(c->pi_coef, 0, n * sizeof(Fr), ctx->stream));
    TP_CUDA_OK(ctx, cudaMemsetAsync(c->buf4[4], 0, 4 * n * sizeof(Fr), ctx->stream));
    c->pi_buffers_zero = true;
  } else if (!pi_zero) {
    c->pi_buffers_zero = false;
  }
  // witness + public-input polynomials (proof.rs:50, 105-106)
  static const bool no_intt_shard = getenv("TP_NO_INTT_SHARD") && *getenv("TP_NO_INTT_SHARD") == '1';
  if (col_ready) {
    if (!pi_zero) TP_TRY(ntt_dev(ctx, c->pi_eval, c->pi_coef, c->log_n, true, nullptr));
  } else if (comm_ready(ctx) && !no_intt_shard && n >= 4096) {
    // sharded context: the interpolations are split by column (column j on rank j mod world) and the coefficient
    // vectors exchanged with one group of device broadcasts -- 32 n bytes over NVLink cost less than an inverse NTT
    const Fr* evs[4] = {c->adv_eval[0], c->adv_eval[1], c->adv_eval[2], c->pi_eval};
    Fr* cfs[4] = {c->adv_coef[0], c->adv_coef[1], c->adv_coef[2], c->pi_coef};
    const int ncol = pi_zero ? 3 : 4;
    const Fr* ins[4];
    Fr* outs[4];
    int cnt = 0;
    for (int j = 0; j < ncol; j++)
      if (j % ctx->world == ctx->rank) {
        ins[cnt] = evs[j];
        outs[cnt] = cfs[j];
        cnt++;
      }
    TP_TRY(ntt_batch_dev(ctx, ins, outs, nullptr, cnt, c->log_n, true));
    TP_TRY(comm_group_begin(ctx));
    for (int j = 0; j < ncol; j++) TP_TRY(comm_bcast(ctx, cfs[j], n * sizeof(Fr), j % ctx->world));
    TP_TRY(comm_group_end(ctx));
  } else {
    const Fr* ins[4] = {c->adv_eval[0], c->adv_eval[1], c->adv_eval[2], c->pi_eval};
    Fr* outs[4] = {c->adv_coef[0], c->adv_coef[1], c->adv_coef[2], c->pi_coef};
    TP_TRY(ntt_batch_dev(ctx, ins, outs, nullptr, pi_zero ? 3 : 4, c->log_n, true));
  }
  if (side) TP_TRY(side_cosets(0, 3, first_guess, 0));   // whatever the per-column path above has not queued yet
  // round 1 commitments (proof.rs:107-110)
  uint8_t com[4][TP_G1_BYTES];
  {
    const Fr* sets[3] = {c->adv_coef[0], c->adv_coef[1], c->adv_coef[2]};
    TP_TRY(msm_batch_dev(ctx, srs, sets, 3, n, com));
  }
  HFr beta, gamma;
  tph::challenges2({com[0], com[1], com[2]}, &beta, &gamma);
  // grand product z (proof.rs:117-131); z_closes: the last value, which the reference pops (proof.rs:120), is 1
  bool z_closes = false;
  {
    const Fr* v[3] = {c->adv_eval[0], c->adv_eval[1], c->adv_eval[2]};
    const Fr* idp[3] = {c->id[0], c->id[1], c->id[2]};
    const Fr* sg[3] = {c->sig_eval[0], c->sig_eval[1], c->sig_eval[2]};
    TP_TRY(perm_grand_product_dev(ctx, v, idp, sg, n, to_dev(beta), to_dev(gamma), c->z_eval, &z_closes));
  }
  TP_TRY(ntt_dev(ctx, c->z_eval, c->z_coef, c->log_n, true, nullptr));
  const bool skip0 = z_closes && !ctx->quotient_all_cosets;
  const unsigned first = skip0 ? 1u : 0u;
  if (side) TP_TRY(side_cosets(0, 4, first, 2));   // z on this rank's cosets; a, b, c only where the guess above missed
  TP_TRY(msm_dev(ctx, srs, c->z_coef, n, com[3]));
  HFr alpha, zeta;
  tph::challenges2({com[0], com[1], com[2], com[3]}, &alpha, &zeta);

  // quotient (proof.rs:292-375) on the 4n domain, coset by coset: four coset NTTs, the pointwise numerator, one
  // inverse coset NTT each.  Coset 0 is H itself, where the numerator is zero whenever the witness satisfies the gates
  // (checked above) and the copy constraints (z closes: the permutation line holds at the last row too) -- its
  // interpolant is then known to be zero and the coset is skipped: 15 transforms instead of 20.  A witness that breaks
  // a copy constraint takes all four cosets and gets the reference's floor quotient (proof.rs:373).
  // Sharded over ranks by coset when the context is sharded (comm.cu); every rank then rebuilds t from the interpolants.
  {
    unsigned mine[4];
    int nmine = 0;
    for (unsigned k = first; k < 4; k++)
      if (coset_owner(ctx, shard, first, k) == ctx->rank) mine[nmine++] = k;
    auto owner = [&](unsigned k) { return coset_owner(ctx, shard, first, k); };
    if (side) TP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->side_ev[3], 0));   // everything queued on the side stream
    TP_TRY(queue_cosets(0, 4, first));   // without the side stream: all of them here
    if (!pi_zero) {
      const Fr* ins[4];
      Fr* outs[4];
      const uint64_t* cos[4];
      for (int m = 0; m < nmine; m++) {
        ins[m] = c->pi_coef;
        outs[m] = c->buf4[4] + (size_t)mine[m] * n;
        cos[m] = mine[m] == 0 ? nullptr : gens[mine[m]].v;
      }
      TP_TRY(ntt_batch_dev(ctx, ins, outs, cos, nmine, c->log_n, false));
    }
    QuotientArgs qa;
    for (int i = 0; i < 5; i++) qa.sel4[i] = c->sel4[i];
    for (int i = 0; i < 3; i++) {
      qa.sig4[i] = c->sig4[i];
      qa.adv4[i] = c->buf4[i];
      qa.k[i] = c->k[i];
    }
    qa.z4 = c->buf4[3];
    qa.pi4 = c->buf4[4];
    qa.l0_4 = c->l0_4;
    TP_TRY(ntt_get_twiddles(ctx, c->log_n + 2, &qa.tw4));
    qa.count = 1;
    qa.stride = 0;
    qa.alpha = &alpha;
    qa.beta = &beta;
    qa.gamma = &gamma;
    qa.out = c->buf4[5];
    qa.n = n;
    TP_TRY(quotient_numerator_dev(ctx, qa, mine, nmine));   // proof 0: the items are the cosets themselves
    {
      // out of place into the (now dead) coset slots of buf4[0]; the interpolants are gathered there
      const Fr* ins[4];
      Fr* outs[4];
      const uint64_t* cos[4];
      for (int m = 0; m < nmine; m++) {
        ins[m] = c->buf4[5] + (size_t)mine[m] * n;
        outs[m] = c->buf4[0] + (size_t)mine[m] * n;
        cos[m] = mine[m] == 0 ? nullptr : gens[mine[m]].v;
      }
      TP_TRY(ntt_batch_dev(ctx, ins, outs, cos, nmine, c->log_n, true));
    }
    if (shard) {
      TP_TRY(comm_group_begin(ctx));
      for (unsigned k = first; k < 4; k++) TP_TRY(comm_bcast(ctx, c->buf4[0] + (size_t)k * n, n * sizeof(Fr), owner(k)));
      TP_TRY(comm_group_end(ctx));
    }
    TP_TRY(quotient_combine_dev(ctx, c->buf4[0], n, 0, 1, &skip0, c->t));
  }

  // The three t commitments (proof.rs:175,181) need nothing that follows: with the MSM pipe they are queued now and
  // accumulate while this stream computes the opening polynomials; the opening witnesses follow as two more sub-batches
  // (the five plain openings, then the linearisation's) and one finish collects all nine points.
  const bool piped = msm_pipe_overlaps(ctx, n);
  if (piped) {
    const Fr* sets[3] = {c->t, c->t + n, c->t + 2 * n};
    TP_TRY(msm_pipe_submit(ctx, srs, sets, 3, n));
  }
  // openings (proof.rs:147-163)
  uint8_t wit[6][TP_G1_BYTES];
  tpp::ProofEvals pe;
  HFr omega = omega_for_log(c->log_n);
  // ... together with the three plain evaluations the linearisation needs (proof.rs:416,429): eight
  // recurrences of length n in one batched scan, one read-back.
  {
    const Fr* polys[8] = {c->adv_coef[0], c->adv_coef[1], c->adv_coef[2], c->z_coef, c->z_coef,
                          c->sig_coef[0], c->sig_coef[1], c->pi_coef};
    Fr* quots[8] = {c->q[0], c->q[1], c->q[2], c->q[3], c->q[4], nullptr, nullptr, nullptr};
    Fr points[8];
    for (int i = 0; i < 8; i++) points[i] = to_dev(i == 4 ? zeta * omega : zeta);
    HFr ys[8];
    TP_TRY(poly_open_batch_dev(ctx, polys, n, points, quots, pi_zero ? 7 : 8, ys));
    for (int i = 0; i < 5; i++) pe.ev[i] = ys[i];
    pe.sig_bar[0] = ys[5];
    pe.sig_bar[1] = ys[6];
    pe.pi_bar = pi_zero ? HFr::zero() : ys[7];
  }
  if (piped) {
    const Fr* sets[5] = {c->q[0], c->q[1], c->q[2], c->q[3], c->q[4]};
    TP_TRY(msm_pipe_submit(ctx, srs, sets, 5, n));
  }
  // linearisation (proof.rs:376-439)
  {
    HFr s[tpp::R_TERMS + 1];
    tpp::lin_scalars(c->k, pe, alpha, beta, gamma, zeta, n, s);
    const LinTerm terms[tpp::R_TERMS] = {{c->sel_coef[0], 0}, {c->sel_coef[1], 0}, {c->sel_coef[2], 0},
                                         {c->sel_coef[3], 0}, {c->sel_coef[4], 0}, {c->z_coef, 0},
                                         {c->sig_coef[2], 0}, {c->t, 0}, {c->t + n, 0}, {c->t + 2 * n, 0}};
    TP_TRY(lincomb_dev(ctx, terms, tpp::R_TERMS, s, n, 1, c->r, 0));
  }
  HFr r_bar;
  TP_TRY(poly_open_dev(ctx, c->r, n, to_dev(zeta), c->q[5], &r_bar));
  // the six opening witnesses and the three t commitments (proof.rs:149,162,163,175,181) are
  // independent of one another: one batch of MSMs.  (q[i][n-1] == 0, so length n is exact.)
  uint8_t tcom[3][TP_G1_BYTES];
  if (piped) {
    const Fr* sets[1] = {c->q[5]};
    TP_TRY(msm_pipe_submit(ctx, srs, sets, 1, n));
    uint8_t outs[9][TP_G1_BYTES];
    TP_TRY(msm_pipe_finish(ctx, outs, 9));
    for (int i = 0; i < 3; i++) memcpy(tcom[i], outs[i], TP_G1_BYTES);
    for (int i = 0; i < 6; i++) memcpy(wit[i], outs[3 + i], TP_G1_BYTES);
  } else {
    const Fr* sets[9] = {c->q[0], c->q[1], c->q[2], c->q[3], c->q[4], c->q[5], c->t, c->t + n, c->t + 2 * n};
    uint8_t outs[9][TP_G1_BYTES];
    TP_TRY(msm_batch_dev(ctx, srs, sets, 9, n, outs));
    for (int i = 0; i < 6; i++) memcpy(wit[i], outs[i], TP_G1_BYTES);
    for (int i = 0; i < 3; i++) memcpy(tcom[i], outs[6 + i], TP_G1_BYTES);
  }

  tpp::write_proof(proof_out, com, wit, tcom, pe.ev, zeta, r_bar);
  return TP_OK;
}

int tp_prove_dev(tp_ctx* ctx, tp_circuit* c, const void* const advice_dev[3], const void* public_inputs_dev,
                 uint8_t* proof_out, size_t proof_cap) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  TP_NO_GROUP(ctx, "prove_dev");
  if (!c || !proof_out || !advice_dev || !advice_dev[0] || !advice_dev[1] || !advice_dev[2] || !public_inputs_dev)
    return fail(ctx, TP_ERR_INVALID_ARG, "prove: null argument");
  if (proof_cap < TP_PROOF_FIXED_BYTES) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "prove: proof buffer too small");
  size_t bytes = c->n * sizeof(Fr);
  for (int i = 0; i < 3; i++)
    TP_CUDA_OK(ctx, cudaMemcpyAsync(c->adv_eval[i], advice_dev[i], bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  TP_CUDA_OK(ctx, cudaMemcpyAsync(c->pi_eval, public_inputs_dev, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  return prove_resident(ctx, c, proof_out);
}
// Witness columns (n each) and the first n_public public inputs from host memory; rows n_public..n of the public-input
// column are zero-filled on the device, which is the `public_inputs.resize(self.rows, Fr::zero())` of proof.rs:52-53.
static int prove_from_host(tp_ctx* ctx, tp_circuit* c, const uint64_t* const advice[3], const uint64_t* public_inputs,
                           size_t n_public, uint8_t* proof_out, size_t proof_cap) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !proof_out) return fail(ctx, TP_ERR_INVALID_ARG, "prove: null argument");
  if (proof_cap < TP_PROOF_FIXED_BYTES) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "prove: proof buffer too small");
  if (is_group(ctx)) {   // CompiledCircuit::prove as ONE call (proof.rs:26-57): every rank proves, rank 0's bytes go out
    std::vector<uint8_t> proofs(ctx->children.size() * TP_PROOF_FIXED_BYTES);
    TP_TRY(group_run(ctx, [&](tp_ctx* cc, int r) {
      return prove_from_host(cc, c->parts[r], advice, public_inputs, n_public, &proofs[(size_t)r * TP_PROOF_FIXED_BYTES], TP_PROOF_FIXED_BYTES);
    }));
    memcpy(proof_out, proofs.data(), TP_PROOF_FIXED_BYTES);
    return TP_OK;
  }
  if (n_public > c->n) return fail(ctx, TP_ERR_INVALID_ARG, "prove: more public inputs than rows");
  if (!advice || !advice[0] || !advice[1] || !advice[2] || (n_public && !public_inputs))
    return fail(ctx, TP_ERR_INVALID_ARG, "prove: null argument");
  size_t bytes = c->n * sizeof(Fr);
  const uint64_t* cols[4] = {advice[0], advice[1], advice[2], public_inputs};
  Fr* dst[4] = {c->adv_eval[0], c->adv_eval[1], c->adv_eval[2], c->pi_eval};
  const int ncols = n_public == c->n ? 4 : 3;   // a short public-input vector travels whole, outside the column slices
  if (ncols == 3) {
    if (n_public) TP_TRY(h2d(ctx, c->pi_eval, public_inputs, n_public * sizeof(Fr)));
    TP_CUDA_OK(ctx, cudaMemsetAsync(c->pi_eval + n_public, 0, (c->n - n_public) * sizeof(Fr), ctx->stream));
  }
  const size_t world = (size_t)ctx->world;
  if (comm_ready(ctx) && c->n % world == 0 && c->n / world >= 64) {
    // Sharded upload: every rank holds the same host columns, so each one sends only its row slice over PCIe
    // and the slices are exchanged over NVLink (one all-gather), then scattered into the columns.
    const size_t rows = c->n / world, slice = rows * sizeof(Fr);
    uint8_t* stage = (uint8_t*)c->buf4[0];                       // [rank][column][rows], at most 4n Fr in total
    for (int j = 0; j < ncols; j++)
      TP_TRY(h2d(ctx, stage + ((size_t)ctx->rank * ncols + j) * slice, (const uint8_t*)cols[j] + (size_t)ctx->rank * slice, slice));
    // [rank][column][rows] is exactly what an in-place all-gather of the ranks' blocks leaves behind: one collective
    // (round 2 started with one broadcast per rank in a group)
    TP_TRY(comm_allgather(ctx, stage + (size_t)ctx->rank * ncols * slice, stage, ncols * slice));
    for (int j = 0; j < ncols; j++)
      TP_CUDA_OK(ctx, cudaMemcpy2DAsync(dst[j], slice, stage + (size_t)j * slice, ncols * slice, slice, world,
                                        cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    // single GPU: columns on the copy stream, one event each; the compute stream picks them up one by one
    if (!ctx->copy_stream) {
      TP_CUDA_OK(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
      for (auto& e : ctx->copy_ev) TP_CUDA_OK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    // the buffers may still be read by work queued earlier on the compute stream (the previous proof)
    TP_CUDA_OK(ctx, cudaEventRecord(ctx->copy_ev[3], ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev[3], 0));
    for (int j = 0; j < 3; j++) {
      TP_CUDA_OK(ctx, cudaMemcpyAsync(dst[j], cols[j], bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
      TP_CUDA_OK(ctx, cudaEventRecord(ctx->copy_ev[j], ctx->copy_stream));
    }
    if (ncols == 4) TP_TRY(h2d(ctx, dst[3], cols[3], bytes));   // the full-length public-input column, compute stream
    return prove_resident(ctx, c, proof_out, ctx->copy_ev);
  }
  return prove_resident(ctx, c, proof_out);
}
int tp_prove(tp_ctx* ctx, tp_circuit* c, const uint64_t* const advice[3], const uint64_t* public_inputs,
             uint8_t* proof_out, size_t proof_cap) {
  return prove_from_host(ctx, c, advice, public_inputs, c ? c->n : 0, proof_out, proof_cap);
}
int tp_prove_inputs(tp_ctx* ctx, tp_circuit* c, const uint64_t* const advice[3], const uint64_t* public_inputs,
                    size_t n_public, uint8_t* proof_out, size_t proof_cap) {
  return prove_from_host(ctx, c, advice, public_inputs, n_public, proof_out, proof_cap);
}

// Intermediate polynomials of the LAST proof of this circuit, straight from the prover's device buffers: the parity
// tests compare them one by one with the reference's own functions (quotient_polynomial, linearisation_poly,
// CompiledPermutation::prove), not only through the final proof bytes.
int tp_circuit_read_poly(tp_ctx* ctx, tp_circuit* c, int which, uint64_t* out, size_t cap_elems, size_t* count) {
  if (!ctx) return TP_ERR_INVALID_ARG;
  if (!c || !count) return fail(ctx, TP_ERR_INVALID_ARG, "read_poly: null argument");
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* cc) { return tp_circuit_read_poly(cc, c->parts[0], which, out, cap_elems, count); });
  const size_t n = c->n;
  const Fr* src = nullptr;
  size_t len = 0;
  switch (which) {
    case TP_POLY_QUOTIENT: src = c->t; len = 3 * n; break;
    case TP_POLY_LINEARISATION: src = c->r; len = n; break;
    case TP_POLY_Z_EVALS: src = c->z_eval; len = n + 1; break;
    case TP_POLY_Z: src = c->z_coef; len = n; break;
    case TP_POLY_A: case TP_POLY_B: case TP_POLY_C: src = c->adv_coef[which - TP_POLY_A]; len = n; break;
    default: return fail(ctx, TP_ERR_INVALID_ARG, "read_poly: unknown polynomial id");
  }
  *count = len;
  if (!out) return TP_OK;
  if (cap_elems < len) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "read_poly: output buffer too small");
  return d2h_sync(ctx, out, src, len * sizeof(Fr));
}

// ---- helpers -------------------------------------------------------------------------------------
int tp_measure_imad_peak(tp_ctx* ctx, double* imad_per_s, double* imad_wide_per_s) {
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_measure_imad_peak(c, imad_per_s, imad_wide_per_s); });
  return measure_imad_dev(ctx, imad_per_s, imad_wide_per_s);
}
int tp_selftest(tp_ctx* ctx, int* failures) {
  if (is_group(ctx)) return on_rank0(ctx, [&](tp_ctx* c) { return tp_selftest(c, failures); });
  return selftest_dev(ctx, failures);
}
int tp_stdrng_words(const uint8_t* seed32, uint64_t seed_u64, size_t count, uint32_t* out) {
  if (!out && count) return TP_ERR_INVALID_ARG;
  tph::StdRng rng = seed32 ? tph::StdRng::from_seed(seed32) : tph::StdRng::seed_from_u64(seed_u64);
  for (size_t i = 0; i < count; i++) out[i] = rng.next_u32();
  return TP_OK;
}
#ifndef TP_BUILD_STAMP
#define TP_BUILD_STAMP "unstamped"
#endif
/* sha256 over every source file and compiler flag this library was built from (typlonk_b200/build.py compares it with
 * the sources on disk, so a stale binary is rebuilt instead of being loaded against newer headers) */
const char* tp_build_stamp(void) { return "tp-build-stamp:" TP_BUILD_STAMP; }
int tp_fr_rand_stream(uint64_t seed, size_t count, uint64_t* out) {
  if (!out && count) return TP_ERR_INVALID_ARG;
  tph::StdRng rng = tph::StdRng::seed_from_u64(seed);
  for (size_t i = 0; i < count; i++) {
    HFr x = tph::fr_rand(rng);
    memcpy(out + 4 * i, x.v, 32);
  }
  return TP_OK;
}

}  // extern "C"
