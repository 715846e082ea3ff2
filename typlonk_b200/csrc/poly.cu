// Elementwise and scan kernels of the prover (all HBM-streaming integer work over Fr):
//   * permutation grand product   -- permutation/src/proving.rs:7-31 (one inversion per cell in
//     the reference) as a prefix-product scan of the numerators and a suffix-product scan of the
//     denominators sharing their launches, with ONE inversion per proof
//   * opening polynomial          -- kzg/src/lib.rs:55-64: Horner evaluation and the division
//     by (X - z) are one linear recurrence q[k-1] = p[k] + z q[k], solved as a hierarchical scan
//   * gate check                  -- the `vanishes(line1)` assert, plonk/src/proof.rs:317-321
//   * quotient numerator on the 4n domain and division by X^n - 1 -- plonk/src/proof.rs:292-375
//     (the reference builds these with O(n^2) `naive_mul`)
//   * linear combination for r(X) -- plonk/src/proof.rs:376-439
//   * sigma / id tables           -- permutation/src/lib.rs:101-128
#include "common.cuh"

namespace tp {

// Element-wise kernels with many field products (the quotient numerator has ~30) are straight-line code far larger than
// the instruction cache; with TP_POLY_MUL_CALL they go through one shared copy of the multiplier (A/B in profiles/).
#ifdef TP_POLY_MUL_CALL
static __device__ __noinline__ Fr pmul(Fr a, Fr b) { return fr_mul(a, b); }
#else
__device__ __forceinline__ Fr pmul(const Fr& a, const Fr& b) { return fr_mul(a, b); }
#endif


// Small per-launch parameter blocks (per-proof scalars, item lists, pointer tables) go through a ring of pinned staging
// blocks, each copied in stream order to a device block of its own.  A staging block is written again only after the
// copy out of it has run, which the stream has long done by then (every stage of a proof ends in a host read-back).
int params_upload(tp_ctx* ctx, const void* src, size_t bytes, const void** dev) {
  const unsigned s = ctx->param_next++ % TP_PARAM_SLOTS;
  if (!ctx->param_ev[s]) TP_CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->param_ev[s], cudaEventDisableTiming));
  TP_CUDA_OK(ctx, cudaEventSynchronize(ctx->param_ev[s]));
  if (ctx->param_host_cap[s] < bytes) {
    if (ctx->param_host[s]) cudaFreeHost(ctx->param_host[s]);
    ctx->param_host[s] = nullptr;
    ctx->param_host_cap[s] = 0;
    const size_t want = bytes < 4096 ? 4096 : bytes;
    TP_CUDA_OK(ctx, cudaMallocHost(&ctx->param_host[s], want));
    ctx->param_host_cap[s] = want;
  }
  TP_TRY(ensure(ctx, ctx->param_dev[s], bytes));
  memcpy(ctx->param_host[s], src, bytes);
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->param_dev[s].p, ctx->param_host[s], bytes, cudaMemcpyHostToDevice, ctx->stream));
  TP_CUDA_OK(ctx, cudaEventRecord(ctx->param_ev[s], ctx->stream));
  *dev = ctx->param_dev[s].p;
  return TP_OK;
}

#define EW_THREADS 256
static inline unsigned ew_grid(size_t n) { return (unsigned)((n + EW_THREADS - 1) / EW_THREADS); }

// =====================================================================================
// exclusive prefix-product scan (in place).  chunk per thread, recursive on chunk totals.
// =====================================================================================
#define SCAN_CH 32
#define SCAN_BASE 64

// 2 * count independent scans of the same length side by side (blockIdx.y = 2 * proof + which): the upper levels of a
// scan are chains of small launches, so the two scans of every proof of a batch cost what one costs.  Scan (proof p,
// which w) runs over a[w] + p * stride; its chunk totals go to tot[w] + p * tot_stride.
struct ScanPair {
  Fr* a[2];
  Fr* tot[2];
  size_t stride, tot_stride;
  __device__ __forceinline__ Fr* arr(unsigned y) const { return ((y & 1) ? a[1] : a[0]) + (size_t)(y >> 1) * stride; }
  __device__ __forceinline__ Fr* tots(unsigned y) const { return ((y & 1) ? tot[1] : tot[0]) + (size_t)(y >> 1) * tot_stride; }
};
__global__ void k_mulscan2_serial(ScanPair p, size_t n) {   // exclusive
  if (threadIdx.x != 0) return;
  Fr* a = p.arr(blockIdx.x);
  Fr acc = fr_one();
  for (size_t i = 0; i < n; i++) {
    Fr x = fr_load(a + i);
    fr_store(a + i, acc);
    acc = fr_mul(acc, x);
  }
}
__global__ void k_mulscan2_chunk(ScanPair p, size_t n) {    // exclusive
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * SCAN_CH;
  if (lo >= n) return;
  Fr* a = p.arr(blockIdx.y);
  size_t hi = lo + SCAN_CH < n ? lo + SCAN_CH : n;
  Fr acc = fr_one();
  for (size_t i = lo; i < hi; i++) {
    Fr x = fr_load(a + i);
    fr_store(a + i, acc);
    acc = fr_mul(acc, x);
  }
  fr_store(p.tots(blockIdx.y) + t, acc);
}
__global__ void k_mulscan2_apply(ScanPair p, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  size_t ch = i / SCAN_CH;
  if (ch == 0) return;
  Fr* a = p.arr(blockIdx.y);
  fr_store(a + i, fr_mul(fr_load(a + i), fr_load(p.tots(blockIdx.y) + ch)));
}
// exclusive prefix products of a0 + p * stride and a1 + p * stride over [0, n), p < count, in place
static int mulscan2_exclusive(tp_ctx* ctx, Fr* a0, Fr* a1, size_t stride, int count, size_t n, int level) {
  ScanPair p;
  p.a[0] = a0;
  p.a[1] = a1;
  p.stride = stride;
  p.tot[0] = p.tot[1] = nullptr;
  p.tot_stride = 0;
  if (n <= SCAN_BASE) {
    k_mulscan2_serial<<<2 * count, 32, 0, ctx->stream>>>(p, n);
    TP_LAUNCH(ctx, "k_mulscan2_serial");
    return TP_OK;
  }
  size_t nch = (n + SCAN_CH - 1) / SCAN_CH;
  TP_TRY(ensure(ctx, ctx->scan_tmp[level], 2 * nch * (size_t)count * sizeof(Fr)));
  p.tot[0] = (Fr*)ctx->scan_tmp[level].p;
  p.tot[1] = p.tot[0] + nch;
  p.tot_stride = 2 * nch;
  k_mulscan2_chunk<<<dim3(ew_grid(nch), 2 * count), EW_THREADS, 0, ctx->stream>>>(p, n);
  TP_LAUNCH(ctx, "k_mulscan2_chunk");
  TP_TRY(mulscan2_exclusive(ctx, p.tot[0], p.tot[1], p.tot_stride, count, nch, level + 1));
  k_mulscan2_apply<<<dim3(ew_grid(n), 2 * count), EW_THREADS, 0, ctx->stream>>>(p, n);
  TP_LAUNCH(ctx, "k_mulscan2_apply");
  return TP_OK;
}

// =====================================================================================
// grand product  (permutation/src/proving.rs:7-31)
// =====================================================================================
// z[0] = 1, z[j+1] = prod_{k<=j} num_k / den_k with num_k = prod_i (v_ik + beta id_ik + gamma), den_k likewise over
// sigma.  The reference inverts every denominator; here NOTHING is inverted per element:
//     1 / prod_{k<=j} den_k = Dtot^-1 * prod_{k>j} den_k,
// so z[j+1] = (prefix product of num up to j) * (suffix product of den after j) * Dtot^-1 -- two product scans that
// share their launches and ONE inversion per proof, done by the host between the up- and the down-sweep (it also
// replaces the zero-denominator flag: a zero denominator makes Dtot zero).  About 15 field products per row in all.
// The grand products of `count` proofs run in the same launches, proof p in blockIdx.y, and the host inverts their
// Dtot values with one batch inversion.
#define PERM_CH 16   // rows per thread
struct PermArgs {
  const Fr* v[3];   // proof p's witness column i: v[i] + p * vstride
  size_t vstride;
  const Fr* id[3];
  const Fr* sg[3];
  const Fr* bg;     // per proof: beta, gamma
  const Fr* dinv;   // per proof: Dtot^-1 (k_perm_finish)
  size_t n;
  Fr* pre;     // n per proof: prefix product of num inside the row's chunk (inclusive)
  Fr* den;     // n per proof: den of the row
  Fr* tot;     // 2 (nch + 1) per proof: chunk totals of num, then a trailing one; chunk totals of den in REVERSE chunk
               // order, then a trailing one
  size_t nch;
};
__global__ void __launch_bounds__(128) k_perm_chunks(PermArgs a) {
  // the proof's beta and gamma are read from shared memory at each use: held in registers they would push the row
  // loop past its register budget
  __shared__ Fr bg[2];
  const size_t p = blockIdx.y;
  if (threadIdx.x < 2) bg[threadIdx.x] = fr_load(a.bg + 2 * p + threadIdx.x);
  __syncthreads();
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > a.nch) return;
  if (t == a.nch) {   // the trailing ones: the exclusive scans then leave the grand totals there
    Fr* tot_num = a.tot + p * 2 * (a.nch + 1);
    fr_store(tot_num + a.nch, fr_one());
    fr_store(tot_num + (a.nch + 1) + a.nch, fr_one());
    return;
  }
  const size_t vo = p * a.vstride;
  Fr* const pre = a.pre + p * a.n;
  Fr* const den_out = a.den + p * a.n;
  const size_t lo = t * PERM_CH;
  const size_t hi = lo + PERM_CH < a.n ? lo + PERM_CH : a.n;
  Fr pn = fr_one(), pd = fr_one();
  for (size_t j = lo; j < hi; j++) {
    Fr num, den;
#pragma unroll
    for (int i = 0; i < 3; i++) {
      Fr v = fr_add(fr_load(a.v[i] + vo + j), fr_load(&bg[1]));
      Fr nu = fr_add(v, pmul(fr_load(&bg[0]), fr_load(a.id[i] + j)));
      Fr de = fr_add(v, pmul(fr_load(&bg[0]), fr_load(a.sg[i] + j)));
      num = i == 0 ? nu : pmul(num, nu);
      den = i == 0 ? de : pmul(den, de);
    }
    pn = j == lo ? num : pmul(pn, num);
    pd = j == lo ? den : pmul(pd, den);
    fr_store(pre + j, pn);
    fr_store(den_out + j, den);
  }
  Fr* tot_num = a.tot + p * 2 * (a.nch + 1);
  fr_store(tot_num + t, pn);
  fr_store(tot_num + (a.nch + 1) + (a.nch - 1 - t), pd);
}
// carry_num[t] = product of num over the chunks before t; carry_den[nch-1-t] = product of den over the chunks after t
__global__ void __launch_bounds__(128) k_perm_finish(PermArgs a, Fr* __restrict__ z /* n + 1 per proof */, size_t zstride) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.nch) return;
  const size_t p = blockIdx.y;
  const Fr* tot_num = a.tot + p * 2 * (a.nch + 1);
  const Fr* tot_den = tot_num + (a.nch + 1);
  const Fr* pre = a.pre + p * a.n;
  const Fr* den = a.den + p * a.n;
  z += p * zstride;
  const size_t lo = t * PERM_CH;
  const size_t hi = lo + PERM_CH < a.n ? lo + PERM_CH : a.n;
  if (t == 0) fr_store(z, fr_one());
  Fr k = pmul(pmul(fr_load(tot_num + t), fr_load(tot_den + (a.nch - 1 - t))), fr_load(a.dinv + p));
  // walk the chunk backwards: k = (carries) * Dtot^-1 * product of the chunk's den after row j
  for (size_t j = hi; j-- > lo;) {
    fr_store(z + j + 1, pmul(fr_load(pre + j), k));
    if (j > lo) k = pmul(k, fr_load(den + j));
  }
}

int perm_grand_product_batch_dev(tp_ctx* ctx, const Fr* const values[3], size_t vstride, const Fr* const id[3],
                                 const Fr* const sigma[3], size_t n, int count, const tph::HFr* beta,
                                 const tph::HFr* gamma, Fr* out, size_t ostride, bool* zero_den, bool* closes) {
  ProfScope prof(ctx, TP_PHASE_PERM);
  const size_t nch = (n + PERM_CH - 1) / PERM_CH;
  const size_t cnt = (size_t)count;
  if (2 * cnt * sizeof(Fr) > ctx->pinned_cap) return fail(ctx, TP_ERR_INVALID_ARG, "permutation prove: batch too large");
  TP_TRY(ensure(ctx, ctx->misc[0], cnt * n * sizeof(Fr)));
  TP_TRY(ensure(ctx, ctx->misc[1], cnt * n * sizeof(Fr)));
  TP_TRY(ensure(ctx, ctx->misc[2], cnt * 2 * (nch + 1) * sizeof(Fr)));
  std::vector<Fr> bg(2 * cnt);
  for (size_t p = 0; p < cnt; p++) {
    bg[2 * p] = to_dev(beta[p]);
    bg[2 * p + 1] = to_dev(gamma[p]);
  }
  PermArgs a;
  for (int i = 0; i < 3; i++) {
    a.v[i] = values[i];
    a.id[i] = id[i];
    a.sg[i] = sigma[i];
  }
  a.vstride = vstride;
  TP_TRY(params_upload(ctx, bg.data(), bg.size() * sizeof(Fr), (const void**)&a.bg));
  a.dinv = nullptr;
  a.n = n;
  a.nch = nch;
  a.pre = (Fr*)ctx->misc[0].p;
  a.den = (Fr*)ctx->misc[1].p;
  a.tot = (Fr*)ctx->misc[2].p;
  k_perm_chunks<<<dim3((unsigned)((nch + 1 + 127) / 128), count), 128, 0, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_perm_chunks");
  TP_TRY(mulscan2_exclusive(ctx, a.tot, a.tot + (nch + 1), 2 * (nch + 1), count, nch + 1, 0));
  // the one inversion per proof: Dtot = product of every denominator (the last slot of the reversed den scan); Ntot
  // the product of every numerator.  Both for every proof in one read-back.
  const size_t pitch = 2 * (nch + 1) * sizeof(Fr);
  uint8_t* host = (uint8_t*)ctx->pinned;
  TP_CUDA_OK(ctx, cudaMemcpy2DAsync(host, sizeof(Fr), a.tot + (2 * nch + 1), pitch, sizeof(Fr), cnt, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaMemcpy2DAsync(host + cnt * sizeof(Fr), sizeof(Fr), a.tot + nch, pitch, sizeof(Fr), cnt, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  std::vector<tph::HFr> dtot(cnt), ntot(cnt), dinv(cnt);
  for (size_t p = 0; p < cnt; p++) {
    memcpy(dtot[p].v, host + p * sizeof(Fr), 32);
    memcpy(ntot[p].v, host + (cnt + p) * sizeof(Fr), 32);
  }
  // Montgomery batch inversion over the non-zero Dtot; a zero one leaves its proof with Dtot^-1 = 0
  {
    tph::HFr acc = tph::HFr::one();
    std::vector<tph::HFr> pre(cnt);
    for (size_t p = 0; p < cnt; p++) {
      pre[p] = acc;
      if (!dtot[p].is_zero()) acc = acc * dtot[p];
    }
    tph::HFr inv = acc.inv();
    for (size_t p = cnt; p-- > 0;) {
      if (dtot[p].is_zero()) {
        dinv[p] = tph::HFr::zero();
        continue;
      }
      dinv[p] = inv * pre[p];
      inv = inv * dtot[p];
    }
  }
  std::vector<Fr> dv(cnt);
  for (size_t p = 0; p < cnt; p++) {
    zero_den[p] = dtot[p].is_zero();
    if (closes) closes[p] = !zero_den[p] && ntot[p] * dinv[p] == tph::HFr::one();   // out[n], the value the caller pops (proof.rs:120)
    dv[p] = to_dev(dinv[p]);
  }
  bool any = false;
  for (size_t p = 0; p < cnt; p++) any = any || !zero_den[p];
  if (!any) return TP_OK;
  TP_TRY(params_upload(ctx, dv.data(), cnt * sizeof(Fr), (const void**)&a.dinv));
  k_perm_finish<<<dim3((unsigned)((nch + 127) / 128), count), 128, 0, ctx->stream>>>(a, out, ostride);
  TP_LAUNCH(ctx, "k_perm_finish");
  return TP_OK;
}
int perm_grand_product_dev(tp_ctx* ctx, const Fr* const values[3], const Fr* const id[3], const Fr* const sigma[3],
                           size_t n, const Fr& beta, const Fr& gamma, Fr* out, bool* closes) {
  const tph::HFr b = to_host(beta), g = to_host(gamma);
  bool zero = false, cl = false;
  TP_TRY(perm_grand_product_batch_dev(ctx, values, 0, id, sigma, n, 1, &b, &g, out, 0, &zero, &cl));
  if (zero) return fail(ctx, TP_ERR_ZERO_DENOMINATOR, "permutation prove: zero denominator");
  if (closes) *closes = cl;
  return TP_OK;
}

// =====================================================================================
// linear recurrence  q[k-1] = p[k] + z q[k]   (Horner + division by X - z)
// =====================================================================================
#define LIN_CH 32
#define LIN_BASE 64
// Any number of independent recurrences of the same length run side by side (blockIdx.y): the scans are latency-bound
// chains of small launches, so the eight evaluations / openings of a proof at its Fiat-Shamir points -- or those of
// every proof of a batch -- cost what one costs.  One level of the hierarchy:
struct LinLevel {
  const Fr* const* p;   // level 0: device table of the inputs (null above level 0)
  Fr* const* q;         // level 0: device table of the quotients (entries may be null: evaluation only)
  const Fr* pbase;      // above level 0: recurrence b's input at pbase + b * stride ...
  Fr* qbase;            // ... and its quotient at qbase + b * stride, where wantq[b]
  size_t stride;
  const unsigned* wantq;
  const Fr* z;          // per recurrence: its point raised to LIN_CH^level
  __device__ __forceinline__ const Fr* in(unsigned b) const { return p ? p[b] : pbase + b * stride; }
  __device__ __forceinline__ Fr* out(unsigned b) const { return q ? q[b] : (wantq[b] ? qbase + b * stride : nullptr); }
};

// h[t] = sum_{k in chunk t} p[k] z^(k - lo)
__global__ void k_linrec_reduce(LinLevel a, size_t n, Fr* h, size_t h_stride) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * LIN_CH;
  if (lo >= n) return;
  const Fr* p = a.in(blockIdx.y);
  const Fr z = fr_load(a.z + blockIdx.y);
  size_t hi = lo + LIN_CH < n ? lo + LIN_CH : n;
  Fr acc = fr_zero();
  for (size_t k = hi; k-- > lo;) acc = fr_add(fr_load(p + k), fr_mul(z, acc));
  fr_store(h + blockIdx.y * h_stride + t, acc);
}
// q[k-1] = p[k] + z q[k] inside chunk t, starting from carry = qprime[t] (q at index hi-1)
__global__ void k_linrec_apply(LinLevel a, size_t n, const Fr* qprime, size_t qp_stride) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * LIN_CH;
  if (lo >= n) return;
  Fr* q = a.out(blockIdx.y);
  if (!q) return;
  const Fr* p = a.in(blockIdx.y);
  const Fr z = fr_load(a.z + blockIdx.y);
  size_t hi = lo + LIN_CH < n ? lo + LIN_CH : n;
  Fr acc = fr_load(qprime + blockIdx.y * qp_stride + t);
  if (hi == n) fr_store(q + n - 1, fr_zero());
  for (size_t k = hi; k-- > lo;) {
    acc = fr_add(fr_load(p + k), fr_mul(z, acc));
    if (k >= 1) fr_store(q + k - 1, acc);
  }
}
// serial base case (one thread per recurrence): q and y = p(z) -> yout[b]
__global__ void k_linrec_serial(LinLevel a, size_t n, unsigned batch, Fr* yout) {
  const unsigned b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const Fr* p = a.in(b);
  Fr* q = a.out(b);
  const Fr z = fr_load(a.z + b);
  Fr acc = fr_zero();
  if (q) fr_store(q + n - 1, fr_zero());
  for (size_t k = n; k-- > 0;) {
    acc = fr_add(fr_load(p + k), fr_mul(z, acc));
    if (q && k >= 1) fr_store(q + k - 1, acc);
  }
  fr_store(yout + b, acc);
}

// y[b] is written to the device words yout[b].
static int linrec(tp_ctx* ctx, const LinLevel& in, int batch, bool any_q, size_t n, Fr* yout, int level) {
  if (n <= LIN_BASE) {
    k_linrec_serial<<<(unsigned)((batch + 63) / 64), 64, 0, ctx->stream>>>(in, n, (unsigned)batch, yout);
    TP_LAUNCH(ctx, "k_linrec_serial");
    return TP_OK;
  }
  size_t nch = (n + LIN_CH - 1) / LIN_CH;
  // level buffers: h (nch per recurrence) and qprime (nch per recurrence)
  TP_TRY(ensure(ctx, ctx->scan_tmp[level], 2 * nch * (size_t)batch * sizeof(Fr)));
  Fr* h = (Fr*)ctx->scan_tmp[level].p;
  Fr* qp = h + nch * batch;
  k_linrec_reduce<<<dim3(ew_grid(nch), (unsigned)batch), EW_THREADS, 0, ctx->stream>>>(in, n, h, nch);
  TP_LAUNCH(ctx, "k_linrec_reduce");
  LinLevel next = in;
  next.p = nullptr;
  next.q = nullptr;
  next.pbase = h;
  next.qbase = qp;
  next.stride = nch;
  next.z = in.z + batch;
  TP_TRY(linrec(ctx, next, batch, any_q, nch, yout, level + 1));
  if (any_q) {
    k_linrec_apply<<<dim3(ew_grid(nch), (unsigned)batch), EW_THREADS, 0, ctx->stream>>>(in, n, qp, nch);
    TP_LAUNCH(ctx, "k_linrec_apply");
  }
  return TP_OK;
}

// Evaluate (and, where q_out[b] is non-null, divide by X - z[b]) `batch` polynomials of `len` coefficients.
int poly_open_batch_dev(tp_ctx* ctx, const Fr* const* p, size_t len, const Fr* z, Fr* const* q_out, int batch,
                        tph::HFr* y) {
  if (len == 0) return fail(ctx, TP_ERR_EMPTY_POLY, "open: empty polynomial");
  if (batch < 1 || batch > 65535 || (size_t)batch * sizeof(Fr) > ctx->pinned_cap)
    return fail(ctx, TP_ERR_INVALID_ARG, "open: bad batch size");
  ProfScope prof(ctx, TP_PHASE_SCAN);
  const size_t nb = (size_t)batch;
  TP_TRY(ensure(ctx, ctx->misc[2], nb * sizeof(Fr)));
  Fr* yd = (Fr*)ctx->misc[2].p;
  // one parameter block: the points of every level, the input and quotient tables, the wanted-quotient flags
  int levels = 1;
  for (size_t m = len; m > LIN_BASE; m = (m + LIN_CH - 1) / LIN_CH) levels++;
  const size_t zbytes = (size_t)levels * nb * sizeof(Fr), pbytes = nb * sizeof(void*);
  std::vector<uint8_t> blk(zbytes + 2 * pbytes + nb * sizeof(unsigned));
  Fr* zs = (Fr*)blk.data();
  const Fr** ps = (const Fr**)(blk.data() + zbytes);
  Fr** qs = (Fr**)(blk.data() + zbytes + pbytes);
  unsigned* wq = (unsigned*)(blk.data() + zbytes + 2 * pbytes);
  bool any_q = false;
  for (size_t b = 0; b < nb; b++) {
    tph::HFr zl = to_host(z[b]);
    for (int l = 0; l < levels; l++) {
      zs[(size_t)l * nb + b] = to_dev(zl);
      zl = zl.pow_u64(LIN_CH);
    }
    ps[b] = p[b];
    qs[b] = q_out ? q_out[b] : nullptr;
    wq[b] = qs[b] ? 1u : 0u;
    any_q = any_q || qs[b];
  }
  const uint8_t* dev = nullptr;
  TP_TRY(params_upload(ctx, blk.data(), blk.size(), (const void**)&dev));
  LinLevel in;
  in.z = (const Fr*)dev;
  in.p = (const Fr* const*)(dev + zbytes);
  in.q = (Fr* const*)(dev + zbytes + pbytes);
  in.wantq = (const unsigned*)(dev + zbytes + 2 * pbytes);
  in.pbase = nullptr;
  in.qbase = nullptr;
  in.stride = 0;
  TP_TRY(linrec(ctx, in, batch, any_q, len, yd, 0));
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->pinned, yd, nb * sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  for (size_t b = 0; b < nb; b++) memcpy(y[b].v, (const uint8_t*)ctx->pinned + 32 * b, 32);
  return TP_OK;
}
int poly_open_dev(tp_ctx* ctx, const Fr* p, size_t len, const Fr& z, Fr* q_out, tph::HFr* y) {
  const Fr* ps[1] = {p};
  Fr* qs[1] = {q_out};
  return poly_open_batch_dev(ctx, ps, len, &z, qs, 1, y);
}

// =====================================================================================
// gate check on the n rows
// =====================================================================================
struct GateArgs {
  const Fr* sel[5];
  const Fr* adv[3];   // proof p (blockIdx.y): adv[i] + p * stride, pi + p * stride
  const Fr* pi;
  size_t n, stride;
  unsigned* flag;     // one per proof
};
__global__ void k_gate_check(GateArgs g) {
  size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= g.n) return;
  const size_t o = (size_t)blockIdx.y * g.stride + j;
  Fr a = fr_load(g.adv[0] + o), b = fr_load(g.adv[1] + o), c = fr_load(g.adv[2] + o);
  Fr acc = fr_mul(fr_load(g.sel[0] + j), a);
  acc = fr_add(acc, fr_mul(fr_load(g.sel[1] + j), b));
  acc = fr_sub(acc, fr_mul(fr_load(g.sel[2] + j), c));
  acc = fr_add(acc, fr_mul(fr_mul(fr_load(g.sel[3] + j), a), b));
  acc = fr_add(acc, fr_load(g.sel[4] + j));
  const Fr pi = fr_load(g.pi + o);
  acc = fr_add(acc, pi);
  // bit 0: the gate equation fails on some row; bit 1: some public input is non-zero
  const unsigned f = (fr_is_zero(acc) ? 0u : 1u) | (fr_is_zero(pi) ? 0u : 2u);
  if (f) atomicOr(g.flag + blockIdx.y, f);
}
int gate_check_dev(tp_ctx* ctx, const Fr* const sel_evals[5], const Fr* const adv[3], const Fr* pi, size_t n,
                   size_t stride, int count, unsigned* flags) {
  const size_t bytes = (size_t)count * sizeof(unsigned);
  if (bytes > ctx->pinned_cap) return fail(ctx, TP_ERR_INVALID_ARG, "gate check: batch too large");
  TP_TRY(ensure(ctx, ctx->flag, bytes));
  GateArgs g;
  for (int i = 0; i < 5; i++) g.sel[i] = sel_evals[i];
  for (int i = 0; i < 3; i++) g.adv[i] = adv[i];
  g.pi = pi;
  g.n = n;
  g.stride = stride;
  g.flag = (unsigned*)ctx->flag.p;
  TP_CUDA_OK(ctx, cudaMemsetAsync(g.flag, 0, bytes, ctx->stream));
  k_gate_check<<<dim3(ew_grid(n), count), EW_THREADS, 0, ctx->stream>>>(g);
  TP_LAUNCH(ctx, "k_gate_check");
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->pinned, g.flag, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(flags, ctx->pinned, bytes);
  return TP_OK;
}

// =====================================================================================
// quotient numerator on the 4n domain, one coset of H at a time
// =====================================================================================
// The 4n-point domain <omega_4n> is the union of the four cosets omega_4n^k H, k = 0..3.  Every
// 4n-sized table here is COSET-MAJOR: entry k * n + i belongs to the point omega_4n^(4i + k).  A
// coset is a self-contained unit of work (five size-n coset NTTs, this kernel, one inverse coset
// NTT), which is what lets the quotient be sharded over GPUs by coset (api.cu).
struct QuotScalars {   // per proof
  Fr alpha, alpha2, beta, gamma;
  Fr bk[3];  // beta * k_i
};
struct QuotKernelArgs {
  const Fr* sel4[5];
  const Fr* sig4[3];
  const Fr* l0_4;
  const Fr* tw4;
  const Fr* adv4[3];   // proof p: + p * stride, likewise z4, pi4 and out
  const Fr* z4;
  const Fr* pi4;
  Fr* out;
  size_t stride;
  const QuotScalars* sc;
  const unsigned* items;   // blockIdx.y selects the item: proof << 2 | coset
  size_t n;
};
__global__ void __launch_bounds__(EW_THREADS) k_quotient_numerator(QuotKernelArgs q) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= q.n) return;
  const unsigned item = q.items[blockIdx.y];
  const unsigned k = item & 3u;
  const size_t po = (size_t)(item >> 2) * q.stride;
  const QuotScalars* sc = q.sc + (item >> 2);
  const size_t half = q.n * 2;
  const size_t i4 = 4 * i + k;               // exponent of omega_4n at this point
  const size_t o = (size_t)k * q.n + i;      // coset-major slot
  Fr x = i4 < half ? fr_load(q.tw4 + i4) : fr_neg(fr_load(q.tw4 + (i4 - half)));
  Fr a = fr_load(q.adv4[0] + po + o), b = fr_load(q.adv4[1] + po + o), c = fr_load(q.adv4[2] + po + o);
  Fr z = fr_load(q.z4 + po + o);
  Fr zw = fr_load(q.z4 + po + (size_t)k * q.n + (i + 1 < q.n ? i + 1 : 0));   // z(omega x): next point of the same coset
  // gate line (proof.rs:317-320)
  Fr acc = pmul(fr_load(q.sel4[0] + o), a);
  acc = fr_add(acc, pmul(fr_load(q.sel4[1] + o), b));
  acc = fr_sub(acc, pmul(fr_load(q.sel4[2] + o), c));
  acc = fr_add(acc, pmul(pmul(fr_load(q.sel4[3] + o), a), b));
  acc = fr_add(acc, fr_load(q.sel4[4] + o));
  acc = fr_add(acc, fr_load(q.pi4 + po + o));
  // permutation lines (proof.rs:323-354)
  const Fr gamma = fr_load(&sc->gamma), beta = fr_load(&sc->beta);
  Fr ag = fr_add(a, gamma), bg = fr_add(b, gamma), cg = fr_add(c, gamma);
  Fr l2 = pmul(fr_add(ag, pmul(fr_load(&sc->bk[0]), x)), fr_add(bg, pmul(fr_load(&sc->bk[1]), x)));
  l2 = pmul(l2, fr_add(cg, pmul(fr_load(&sc->bk[2]), x)));
  l2 = pmul(l2, z);
  Fr l3 = pmul(fr_add(ag, pmul(beta, fr_load(q.sig4[0] + o))), fr_add(bg, pmul(beta, fr_load(q.sig4[1] + o))));
  l3 = pmul(l3, fr_add(cg, pmul(beta, fr_load(q.sig4[2] + o))));
  l3 = pmul(l3, zw);
  acc = fr_add(acc, pmul(fr_load(&sc->alpha), fr_sub(l2, l3)));
  // L0 line (proof.rs:355-360)
  Fr l4 = pmul(fr_sub(z, fr_one()), fr_load(q.l0_4 + o));
  acc = fr_add(acc, pmul(fr_load(&sc->alpha2), l4));
  fr_store(q.out + po + o, acc);
}
int quotient_numerator_dev(tp_ctx* ctx, const QuotientArgs& a, const unsigned* items, int nitems) {
  if (nitems <= 0) return TP_OK;
  if (nitems > 65535) return fail(ctx, TP_ERR_INVALID_ARG, "quotient: too many cosets in one launch");
  ProfScope prof(ctx, TP_PHASE_QUOTIENT);
  QuotKernelArgs q;
  for (int i = 0; i < 5; i++) q.sel4[i] = a.sel4[i];
  for (int i = 0; i < 3; i++) {
    q.sig4[i] = a.sig4[i];
    q.adv4[i] = a.adv4[i];
  }
  q.z4 = a.z4;
  q.pi4 = a.pi4;
  q.l0_4 = a.l0_4;
  q.tw4 = a.tw4;
  q.out = a.out;
  q.stride = a.stride;
  q.n = a.n;
  // one parameter block: the per-proof scalars, then the items
  const size_t sbytes = (size_t)a.count * sizeof(QuotScalars);
  std::vector<uint8_t> blk(sbytes + (size_t)nitems * sizeof(unsigned));
  QuotScalars* sc = (QuotScalars*)blk.data();
  for (int p = 0; p < a.count; p++) {
    sc[p].alpha = to_dev(a.alpha[p]);
    sc[p].alpha2 = to_dev(a.alpha[p].sqr());
    sc[p].beta = to_dev(a.beta[p]);
    sc[p].gamma = to_dev(a.gamma[p]);
    for (int i = 0; i < 3; i++) sc[p].bk[i] = to_dev(a.beta[p] * a.k[i]);
  }
  memcpy(blk.data() + sbytes, items, (size_t)nitems * sizeof(unsigned));
  const uint8_t* dev = nullptr;
  TP_TRY(params_upload(ctx, blk.data(), blk.size(), (const void**)&dev));
  q.sc = (const QuotScalars*)dev;
  q.items = (const unsigned*)(dev + sbytes);
  k_quotient_numerator<<<dim3(ew_grid(a.n), (unsigned)nitems), EW_THREADS, 0, ctx->stream>>>(q);
  TP_LAUNCH(ctx, "k_quotient_numerator");
  return TP_OK;
}

// Numerator coefficients from its four per-coset interpolants, and the floor division by X^n - 1
// (proof.rs:373, 504-508; the remainder is discarded as the reference does).  Write
// N(X) = sum_j X^(jn) N_j(X), deg N_j < n.  On coset k, x^n = iota^k (iota = omega_4n^n, iota^2 = -1),
// so the interpolant of coset k is C_k = sum_j iota^(kj) N_j and N_j = 1/4 sum_k iota^(-kj) C_k.
// Then t_2 = N_3, t_1 = N_2 + t_2, t_0 = N_1 + t_1.
// c0_is_zero: the numerator vanishes on H itself (always, for a witness that satisfies the copy constraints), so
// coset 0 was never evaluated and its slot holds nothing.
// Proof p (blockIdx.y) reads c4 + p * stride and writes t + p * stride.
__global__ void k_quotient_combine(const Fr* __restrict__ c4, size_t n, size_t stride, Fr iota_inv, Fr quarter,
                                   const unsigned* __restrict__ c0_is_zero, Fr* __restrict__ t) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  c4 += blockIdx.y * stride;
  t += blockIdx.y * stride;
  const Fr c0 = c0_is_zero[blockIdx.y] ? fr_zero() : fr_load(c4 + i);
  const Fr c1 = fr_load(c4 + n + i), c2 = fr_load(c4 + 2 * n + i), c3 = fr_load(c4 + 3 * n + i);
  const Fr e = fr_add(c0, c2), f = fr_sub(c0, c2), g = fr_add(c1, c3);
  const Fr h = fr_mul(iota_inv, fr_sub(c1, c3));
  const Fr n1 = fr_mul(quarter, fr_add(f, h));
  const Fr n2 = fr_mul(quarter, fr_sub(e, g));
  const Fr n3 = fr_mul(quarter, fr_sub(f, h));
  const Fr t1 = fr_add(n2, n3);
  fr_store(t + 2 * n + i, n3);
  fr_store(t + n + i, t1);
  fr_store(t + i, fr_add(n1, t1));
}
int quotient_combine_dev(tp_ctx* ctx, const Fr* c4, size_t n, size_t stride, int count, const bool* c0_is_zero, Fr* t) {
  ProfScope prof(ctx, TP_PHASE_QUOTIENT);
  // iota = omega_4n^n is a primitive fourth root of unity: iota^-1 = -iota; quarter = 4^-1
  unsigned log_n = 0;
  while (((size_t)1 << log_n) < n) log_n++;
  tph::HFr iota_inv = omega_for_log(log_n + 2).pow_u64((uint64_t)n).neg();
  tph::HFr quarter = tph::HFr::from_u64(4).inv();
  std::vector<unsigned> flags(count);
  for (int p = 0; p < count; p++) flags[p] = c0_is_zero[p] ? 1u : 0u;
  const unsigned* fd = nullptr;
  TP_TRY(params_upload(ctx, flags.data(), flags.size() * sizeof(unsigned), (const void**)&fd));
  k_quotient_combine<<<dim3(ew_grid(n), count), EW_THREADS, 0, ctx->stream>>>(c4, n, stride, to_dev(iota_inv), to_dev(quarter), fd, t);
  TP_LAUNCH(ctx, "k_quotient_combine");
  return TP_OK;
}

// L0(x) = (x^n - 1) / (n (x - 1)) on the 4n domain (coset-major output); chunked batch inversion (8 per thread).
#define L0_CH 8
__global__ void k_l0_evals(const Fr* tw4, size_t n, Fr ninv, Fr* out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t n4 = 4 * n, half = 2 * n;
  size_t lo = t * L0_CH;
  if (lo >= n4) return;
  Fr xs[L0_CH], pre[L0_CH];
  Fr acc = fr_one();
  Fr one = fr_one();
  for (int i = 0; i < L0_CH; i++) {
    size_t idx = lo + i;
    Fr x = idx < half ? fr_load(tw4 + idx) : fr_neg(fr_load(tw4 + (idx - half)));
    Fr d = fr_sub(x, one);
    if ((idx & 3) == 0) d = one;  // x in H: handled separately (avoid the zero at x = 1)
    xs[i] = d;
    pre[i] = acc;
    acc = fr_mul(acc, d);
  }
  Fr inv = fr_inv(acc);
  // x^n = iota^(idx mod 4), iota = omega_4n^n
  Fr iota = fr_load(tw4 + n);
  for (int i = L0_CH - 1; i >= 0; i--) {
    size_t idx = lo + i;
    Fr di = fr_mul(inv, pre[i]);
    inv = fr_mul(inv, xs[i]);
    Fr r;
    unsigned m = (unsigned)(idx & 3);
    if (m == 0) {
      r = idx == 0 ? one : fr_zero();
    } else {
      Fr xn = m == 1 ? iota : (m == 2 ? fr_neg(one) : fr_neg(iota));
      r = fr_mul(fr_mul(fr_sub(xn, one), ninv), di);
    }
    fr_store(out + (size_t)m * n + (idx >> 2), r);
  }
}
int l0_evals_4n_dev(tp_ctx* ctx, const Fr* tw4, size_t n, Fr* out) {
  tph::HFr ninv = tph::HFr::from_u64((uint64_t)n).inv();
  size_t nth = (4 * n + L0_CH - 1) / L0_CH;
  if ((4 * n) % L0_CH != 0) return fail(ctx, TP_ERR_INVALID_ARG, "l0: 4n must be a multiple of 8");
  k_l0_evals<<<(unsigned)((nth + 127) / 128), 128, 0, ctx->stream>>>(tw4, n, to_dev(ninv), out);
  TP_LAUNCH(ctx, "k_l0_evals");
  return TP_OK;
}

// =====================================================================================
// linear combination out = constant (at coeff 0) + sum_t s_t * p_t
// =====================================================================================
#define LIN_MAX_TERMS 12
struct LinArgs {
  const Fr* p[LIN_MAX_TERMS];
  size_t pstride[LIN_MAX_TERMS];   // proof p reads term t at p[t] + p * pstride[t] (0: shared by every proof)
  int nterms;
  const Fr* s;                     // per proof: nterms scalars, then the constant
  size_t n, ostride;
  Fr* out;                         // proof p: out + p * ostride
};
__global__ void k_lincomb(LinArgs a) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const size_t pr = blockIdx.y;
  const Fr* s = a.s + pr * (a.nterms + 1);
  Fr acc = i == 0 ? fr_load(s + a.nterms) : fr_zero();
  for (int t = 0; t < a.nterms; t++) acc = fr_add(acc, fr_mul(fr_load(s + t), fr_load(a.p[t] + pr * a.pstride[t] + i)));
  fr_store(a.out + pr * a.ostride + i, acc);
}
int lincomb_dev(tp_ctx* ctx, const LinTerm* terms, int nterms, const tph::HFr* scalars, size_t n, int count, Fr* out,
                size_t ostride) {
  if (nterms > LIN_MAX_TERMS) return fail(ctx, TP_ERR_INVALID_ARG, "lincomb: too many terms");
  LinArgs a;
  for (int t = 0; t < nterms; t++) {
    a.p[t] = terms[t].p;
    a.pstride[t] = terms[t].stride;
  }
  std::vector<Fr> s((size_t)count * (nterms + 1));
  for (size_t i = 0; i < s.size(); i++) s[i] = to_dev(scalars[i]);
  TP_TRY(params_upload(ctx, s.data(), s.size() * sizeof(Fr), (const void**)&a.s));
  a.nterms = nterms;
  a.n = n;
  a.out = out;
  a.ostride = ostride;
  k_lincomb<<<dim3(ew_grid(n), count), EW_THREADS, 0, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_lincomb");
  return TP_OK;
}

// =====================================================================================
// sigma / id tables
// =====================================================================================
struct SigmaArgs {
  const uint64_t* perm;
  size_t n;
  const Fr* tw;  // omega_n^i, i in [0, n/2]
  Fr k[3];
  Fr* id[3];
  Fr* sg[3];
};
__device__ __forceinline__ Fr root_pow(const Fr* tw, size_t n, size_t j) {
  size_t half = n >> 1;
  if (n == 1) return fr_one();
  return j < half ? fr_load(tw + j) : fr_neg(fr_load(tw + (j - half)));
}
__global__ void k_sigma_tables(SigmaArgs a) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * a.n) return;
  size_t i = idx / a.n, j = idx % a.n;
  uint64_t p = a.perm[idx];
  size_t ti = (size_t)(p / a.n), tj = (size_t)(p % a.n);
  Fr ki = i == 0 ? a.k[0] : (i == 1 ? a.k[1] : a.k[2]);
  Fr kt = ti == 0 ? a.k[0] : (ti == 1 ? a.k[1] : a.k[2]);
  Fr idv = fr_mul(ki, root_pow(a.tw, a.n, j));
  Fr sgv = fr_mul(kt, root_pow(a.tw, a.n, tj));
  Fr* idp = i == 0 ? a.id[0] : (i == 1 ? a.id[1] : a.id[2]);
  Fr* sgp = i == 0 ? a.sg[0] : (i == 1 ? a.sg[1] : a.sg[2]);
  fr_store(idp + j, idv);
  fr_store(sgp + j, sgv);
}
int sigma_tables_dev(tp_ctx* ctx, const uint64_t* perm_dev, size_t n, const Fr* tw, const Fr k[3], Fr* id[3],
                     Fr* sigma[3]) {
  SigmaArgs a;
  a.perm = perm_dev;
  a.n = n;
  a.tw = tw;
  for (int i = 0; i < 3; i++) {
    a.k[i] = k[i];
    a.id[i] = id[i];
    a.sg[i] = sigma[i];
  }
  k_sigma_tables<<<ew_grid(3 * n), EW_THREADS, 0, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_sigma_tables");
  return TP_OK;
}

__global__ void k_pad_copy(const Fr* in, size_t len, Fr* out, size_t out_len) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_len) return;
  uint4* o = reinterpret_cast<uint4*>(out + i);
  if (i < len) {
    const uint4* s = reinterpret_cast<const uint4*>(in + i);
    o[0] = s[0];
    o[1] = s[1];
  } else {
    o[0] = make_uint4(0, 0, 0, 0);
    o[1] = make_uint4(0, 0, 0, 0);
  }
}
int pad_copy_dev(tp_ctx* ctx, const Fr* in, size_t len, Fr* out, size_t out_len) {
  k_pad_copy<<<ew_grid(out_len), EW_THREADS, 0, ctx->stream>>>(in, len, out, out_len);
  TP_LAUNCH(ctx, "k_pad_copy");
  return TP_OK;
}
__global__ void k_rotate_copy(const Fr* in, size_t n, size_t shift, Fr* out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  size_t s = i + shift;
  if (s >= n) s -= n;
  const uint4* src = reinterpret_cast<const uint4*>(in + s);
  uint4* o = reinterpret_cast<uint4*>(out + i);
  o[0] = src[0];
  o[1] = src[1];
}
int rotate_copy_dev(tp_ctx* ctx, const Fr* in, size_t n, size_t shift, Fr* out) {
  k_rotate_copy<<<ew_grid(n), EW_THREADS, 0, ctx->stream>>>(in, n, shift % n, out);
  TP_LAUNCH(ctx, "k_rotate_copy");
  return TP_OK;
}

}  // namespace tp
