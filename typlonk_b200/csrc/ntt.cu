// Radix-2 NTT / iNTT / coset NTT over BLS12-381 Fr for sm_100a.
//
// Replaces ark-poly 0.3.0 `Radix2EvaluationDomain::{fft,ifft}_in_place` behind
// `Evaluations::interpolate` / `evaluate_over_domain` (reference call sites
// plonk/src/proof.rs:50,106,115,125,128,337,415; plonk/src/builder.rs:85;
// permutation/src/lib.rs:171,188).  Natural order in, natural order out.
//
// Structure: decimation-in-time with the bit-reversal folded into the first pass's
// gather, ceil(log N / 9) passes over HBM.  A CTA owns a tile of 2^(k+cw) <= 2048 elements
// (2^cw adjacent columns x 2^k rows, rows 2^s0 apart in memory) and runs k butterfly stages on
// it.  Every thread keeps EIGHT elements in registers and does three stages (a radix-8
// butterfly: 12 products, 7 twiddle loads) between two exchanges through shared memory; the
// first round of a pass is loaded straight from global memory and the last one is stored
// straight back, so a 9-stage pass crosses shared memory twice instead of nine times.  The first
// round of the first pass has twiddles 1, w4, w8^q only: the products by 1 are skipped (4 instead
// of 12).  Shared memory holds two uint4 planes with an XOR swizzle (slot i -> i ^ ((i >> 3) & 7))
// that makes every exchange conflict-free for every round geometry.  Twiddles come from one
// table omega_N^i, i in [0, N/2]; the inverse transform reads the same table mirrored
// (omega^-i = -omega^(N/2-i)) so no second table is kept.  Coset scaling uses one table
// scale * g^i per (size, generator), applied at the first load / last store (one product).
#include "common.cuh"

namespace tp {

static const uint64_t ROOT_OF_UNITY_CANON[4] = {0x3829971f439f0d2bull, 0xb63683508c2280b9ull, 0xd09b681922c813b4ull,
                                                0x16a2a19edfe81f20ull};  // 7^((r-1)/2^32)

tph::HFr omega_for_log(unsigned log_n) {
  tph::HFr w = tph::HFr::to_mont(ROOT_OF_UNITY_CANON);
  for (unsigned i = log_n; i < 32; i++) w = w.sqr();
  return w;
}

// out[i] = base^(i * stride_exp) ... generic power table: out[i] = base^i for i < count.
__global__ void k_pow_table(Fr* out, Fr base, size_t count, Fr scale) {
  const int PER = 16;
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t start = t * PER;
  if (start >= count) return;
  Fr cur = fr_mul(scale, fr_pow_u64(base, (unsigned long long)start));
  for (int i = 0; i < PER && start + i < count; i++) {
    fr_store(out + start + i, cur);
    cur = fr_mul(cur, base);
  }
}

int pow_table_dev(tp_ctx* ctx, Fr* out, const tph::HFr& base, size_t count) {
  if (count == 0) return TP_OK;
  k_pow_table<<<(unsigned)(((count + 15) / 16 + 127) / 128), 128, 0, ctx->stream>>>(out, to_dev(base), count,
                                                                                   to_dev(tph::HFr::one()));
  TP_LAUNCH(ctx, "k_pow_table");
  return TP_OK;
}

__device__ __forceinline__ unsigned bitrev(unsigned x, unsigned bits) { return bits == 0 ? 0u : (__brev(x) >> (32 - bits)); }

// Up to NTT_MAX_BATCH transforms of the same size and direction run in one launch (blockIdx.y):
// the prover's 20 coset NTTs of a proof fill whole waves of CTAs instead of one and a half each.
#define NTT_MAX_BATCH 20
struct NttPassArgs {
  const Fr* in[NTT_MAX_BATCH];
  Fr* out[NTT_MAX_BATCH];
  const Fr* coset[NTT_MAX_BATCH];  // scale * g^i (forward: applied at the first load; inverse: at the last store, n^-1 folded in)
  const Fr* tw;
  unsigned L, s0, k, cw;
  int first, inverse, last;
  Fr ninv;
};

// ---- small transforms (log N < 3) and reference structure: one stage per shared-memory round ----
__global__ void __launch_bounds__(512) k_ntt_small(NttPassArgs a) {
  __shared__ uint4 s_lo[8];
  __shared__ uint4 s_hi[8];
  const unsigned T = 1u << a.k;
  const Fr* in = a.in[blockIdx.y];   // may alias out (later passes run in place)
  Fr* out = a.out[blockIdx.y];
  const Fr* coset = a.coset[blockIdx.y];
  for (unsigned e = threadIdx.x; e < T; e += blockDim.x) {
    Fr x = fr_load(in + e);
    if (coset && !a.inverse) x = fr_mul(x, fr_load(coset + e));
    unsigned spos = bitrev(e, a.k);
    s_lo[spos] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    s_hi[spos] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
  }
  __syncthreads();
  const unsigned half_n = 1u << (a.L - 1);
  for (unsigned t = 1; t <= a.k; t++) {
    for (unsigned b = threadIdx.x; b < (T >> 1); b += blockDim.x) {
      unsigned j = b & ((1u << (t - 1)) - 1);
      unsigned p0 = ((b >> (t - 1)) << t) + j, p1 = p0 + (1u << (t - 1));
      unsigned idx = j << (a.L - t);
      Fr w = fr_load(a.tw + (a.inverse ? (half_n - idx) : idx));
      uint4 ul = s_lo[p0], uh = s_hi[p0], vl = s_lo[p1], vh = s_hi[p1];
      Fr u, v;
      u.v[0] = ul.x; u.v[1] = ul.y; u.v[2] = ul.z; u.v[3] = ul.w; u.v[4] = uh.x; u.v[5] = uh.y; u.v[6] = uh.z; u.v[7] = uh.w;
      v.v[0] = vl.x; v.v[1] = vl.y; v.v[2] = vl.z; v.v[3] = vl.w; v.v[4] = vh.x; v.v[5] = vh.y; v.v[6] = vh.z; v.v[7] = vh.w;
      Fr wv = fr_mul(w, v);
      Fr r0 = a.inverse ? fr_sub(u, wv) : fr_add(u, wv);
      Fr r1 = a.inverse ? fr_add(u, wv) : fr_sub(u, wv);
      s_lo[p0] = make_uint4(r0.v[0], r0.v[1], r0.v[2], r0.v[3]);
      s_hi[p0] = make_uint4(r0.v[4], r0.v[5], r0.v[6], r0.v[7]);
      s_lo[p1] = make_uint4(r1.v[0], r1.v[1], r1.v[2], r1.v[3]);
      s_hi[p1] = make_uint4(r1.v[4], r1.v[5], r1.v[6], r1.v[7]);
    }
    __syncthreads();
  }
  for (unsigned e = threadIdx.x; e < T; e += blockDim.x) {
    uint4 xl = s_lo[e], xh = s_hi[e];
    Fr x;
    x.v[0] = xl.x; x.v[1] = xl.y; x.v[2] = xl.z; x.v[3] = xl.w; x.v[4] = xh.x; x.v[5] = xh.y; x.v[6] = xh.z; x.v[7] = xh.w;
    if (a.inverse) x = fr_mul(x, coset ? fr_load(coset + e) : a.ninv);
    fr_store(out + e, x);
  }
}

// ---- register radix-8 passes ---------------------------------------------------------------
// Tile coordinates: row m in [0, 2^k) (the dimension the butterflies run along), column l in
// [0, 2^cw).  Slot of (m, l) in shared memory = swizzle((m << cw) | l).  In a round with field
// base f a thread owns the eight rows m = (m_hi << (f + 3)) | (e << f) | m_lo, e = 0..7, of one
// column; stage bit beta = f + d pairs e with e ^ (1 << d).  Global stage s = s0 + beta + 1 uses
// twiddle omega_N^idx, idx = (((m mod 2^beta) << s0) + lo_val) << (L - s), lo_val = position of
// the column inside its 2^s0 block (0 in the first pass).
__device__ __forceinline__ unsigned ntt_swz(unsigned i) { return i ^ ((i >> 3) & 7u); }

// The multiplier is inlined into the butterflies: a kernel instance carries one full round (12 products with eight
// elements per thread) plus the shorter rounds it needs, ~110 KB of SASS, and ptxas may interleave the independent
// butterflies of a stage.  TP_NTT_MUL_CALL routes every product through one shared copy instead (36 KB): faster in
// round 1, when every place a round was used had its own inlined copy (210 KB), 4-9 % slower now
// (profiles/r2_summary.md L).
#ifdef TP_NTT_MUL_CALL
static __device__ __noinline__ Fr ntt_mul(Fr a, Fr b) { return fr_mul(a, b); }
#else
__device__ __forceinline__ Fr ntt_mul(const Fr& a, const Fr& b) { return fr_mul(a, b); }
#endif
// Lazy butterflies (default; -DTP_NTT_NO_LAZY restores canonical values throughout: 3-4.5 % slower, profiles/r2_summary.md L):
// the values a transform carries between its first load and its last store live in [0, 2r) -- the
// twiddle product skips its final conditional subtraction (fr_mul_lazy: reduced twiddle first, lazy value second), sums
// and differences are reduced modulo 2r, the last store normalises (forward) or multiplies by n^-1 / the coset table
// with a full reduction (inverse).  Saves the product's 17-instruction subtraction per butterfly.
#ifndef TP_NTT_NO_LAZY
__device__ __forceinline__ Fr bf_mul(const Fr& w, const Fr& x) { return fr_mul_lazy(w, x); }
__device__ __forceinline__ Fr bf_add(const Fr& a, const Fr& b) { return fr_add2(a, b); }
__device__ __forceinline__ Fr bf_sub(const Fr& a, const Fr& b) { return fr_sub2(a, b); }
__device__ __forceinline__ Fr bf_out(const Fr& a) { return fr_norm2(a); }
#else
__device__ __forceinline__ Fr bf_mul(const Fr& w, const Fr& x) { return ntt_mul(w, x); }
__device__ __forceinline__ Fr bf_add(const Fr& a, const Fr& b) { return fr_add(a, b); }
__device__ __forceinline__ Fr bf_sub(const Fr& a, const Fr& b) { return fr_sub(a, b); }
__device__ __forceinline__ Fr bf_out(const Fr& a) { return a; }
#endif

// One round = B butterfly stages on the E = 2^B elements a thread holds in registers.
template <int B, int D0, int NST, bool TRIV, bool INVERSE>
__device__ __forceinline__ void ntt_round(Fr (&x)[1 << B], const Fr* __restrict__ tw, unsigned A, unsigned sh, unsigned L,
                                          unsigned half_n) {
  constexpr int E = 1 << B;
#pragma unroll
  for (int d = D0; d < D0 + NST; d++) {
    const unsigned base_idx = A << (sh - d);
#pragma unroll
    for (int e0 = 0; e0 < E; e0++) {
      if (e0 & (1 << d)) continue;
      const int e1 = e0 | (1 << d);
      const unsigned q = e0 & ((1 << d) - 1);
      if (TRIV && q == 0) {  // A == 0 and q == 0: twiddle 1 in both directions
        const Fr u = x[e0], v = x[e1];
        x[e0] = bf_add(u, v);
        x[e1] = bf_sub(u, v);
      } else {
        const unsigned idx = base_idx + (q << (L - d - 1));
        const Fr w = fr_load(tw + (INVERSE ? half_n - idx : idx));
        const Fr t = bf_mul(w, x[e1]);
        const Fr u = x[e0];
        x[e0] = INVERSE ? bf_sub(u, t) : bf_add(u, t);   // mirrored table entry is -omega^-idx
        x[e1] = INVERSE ? bf_add(u, t) : bf_sub(u, t);
      }
    }
  }
}

// Tile = 2^tile_log elements = 256 threads x E: 2048 with eight elements per thread (B = 3: 128 registers, two
// blocks per SM), 1024 with four (B = 2: half the data registers, three blocks per SM -- more warps to cover the
// multiplier's dependent chains, one more trip through shared memory per six stages).
#define NTT_TILE_LOG(B) ((B) == 3 ? 11u : 10u)

// FIRST: first pass of a transform (bit-reversed gather, coset scaling on the way in, trivial twiddles in the first
// round); INVERSE: mirrored twiddles, scaling on the way out.  Compile-time, so that a kernel carries ONE copy of the
// full round in its round loop (the first pass also its cheaper first round) instead of one per place a round is
// used, and no per-limb selects on the direction.
#ifndef TP_NTT_B2_BLOCKS
#define TP_NTT_B2_BLOCKS 3
#endif
template <int B, bool FIRST, bool INVERSE>
__global__ void __launch_bounds__(256, B == 3 ? 2 : TP_NTT_B2_BLOCKS) k_ntt_r8(NttPassArgs a) {
  constexpr int E = 1 << B;
  extern __shared__ uint4 ntt_sh[];
  const unsigned T = 1u << (a.k + a.cw);
  uint4* s_lo = ntt_sh;
  uint4* s_hi = ntt_sh + T;
  const unsigned tau = threadIdx.x;
  const unsigned l = tau & ((1u << a.cw) - 1), rho = tau >> a.cw;
  const unsigned half_n = 1u << (a.L - 1);
  const Fr* in = a.in[blockIdx.y];   // may alias out (later passes run in place)
  Fr* out = a.out[blockIdx.y];
  const Fr* coset = a.coset[blockIdx.y];
  unsigned base = 0, lo_val = 0;
  if (!FIRST) {
    const unsigned hi_idx = blockIdx.x >> (a.s0 - a.cw);
    const unsigned lo_grp = blockIdx.x & ((1u << (a.s0 - a.cw)) - 1);
    base = (hi_idx << (a.s0 + a.k)) + (lo_grp << a.cw) + l;
    lo_val = (lo_grp << a.cw) + l;
  } else {
    base = (blockIdx.x << a.cw) + l;
  }
  Fr x[E];
  const unsigned rem = a.k % B;
  unsigned f_prev = 0;
  for (unsigned f = 0; f < a.k; f += B) {
    const bool tail = f + B > a.k;          // fewer than B stages left: field sits at the top
    const unsigned fb = tail ? a.k - B : f;
    if (f == 0) {
      // ---- first round: operands straight from global memory (field base 0: m = rho * E + e) ----
#pragma unroll
      for (int e = 0; e < E; e++) {
        const unsigned m = (rho << B) | e;
        const unsigned g = FIRST ? (bitrev(m, a.k) << (a.L - a.k)) + base : base + (m << a.s0);
        x[e] = fr_load(in + g);
        if (FIRST && !INVERSE && coset) x[e] = bf_mul(fr_load(coset + g), x[e]);
      }
      if (FIRST) {
        ntt_round<B, 0, B, true, INVERSE>(x, a.tw, 0u, a.L - 1, a.L, half_n);
        continue;
      }
    } else {
      // ---- further rounds: exchange through shared memory ----
      {
        const unsigned m_lo = rho & ((1u << f_prev) - 1), m_hi = rho >> f_prev;
        const unsigned i0 = (((m_hi << (f_prev + B)) | m_lo) << a.cw) | l;
        if (f_prev != 0) __syncthreads();     // the previous exchange has been read by everyone
#pragma unroll
        for (int e = 0; e < E; e++) {
          const unsigned p = ntt_swz(i0 | ((unsigned)e << (f_prev + a.cw)));
          s_lo[p] = make_uint4(x[e].v[0], x[e].v[1], x[e].v[2], x[e].v[3]);
          s_hi[p] = make_uint4(x[e].v[4], x[e].v[5], x[e].v[6], x[e].v[7]);
        }
        __syncthreads();
      }
      const unsigned m_lo = rho & ((1u << fb) - 1), m_hi = rho >> fb;
      const unsigned i0 = (((m_hi << (fb + B)) | m_lo) << a.cw) | l;
#pragma unroll
      for (int e = 0; e < E; e++) {
        const unsigned p = ntt_swz(i0 | ((unsigned)e << (fb + a.cw)));
        const uint4 lo = s_lo[p], hi = s_hi[p];
        x[e].v[0] = lo.x; x[e].v[1] = lo.y; x[e].v[2] = lo.z; x[e].v[3] = lo.w;
        x[e].v[4] = hi.x; x[e].v[5] = hi.y; x[e].v[6] = hi.z; x[e].v[7] = hi.w;
      }
    }
    const unsigned m_lo = rho & ((1u << fb) - 1);
    const unsigned A = (m_lo << a.s0) + lo_val;
    const unsigned sh = a.L - a.s0 - fb - 1;
    if (!tail) {
      ntt_round<B, 0, B, false, INVERSE>(x, a.tw, A, sh, a.L, half_n);
    } else if (rem == 1) {
      ntt_round<B, B - 1, 1, false, INVERSE>(x, a.tw, A, sh, a.L, half_n);
    } else {
      if constexpr (B >= 3) ntt_round<B, B - 2, 2, false, INVERSE>(x, a.tw, A, sh, a.L, half_n);
    }
    f_prev = fb;
  }
  // ---- store from the last round's field ----
  {
    const unsigned m_lo = rho & ((1u << f_prev) - 1), m_hi = rho >> f_prev;
    const unsigned m0 = (m_hi << (f_prev + B)) | m_lo;
    const unsigned obase = FIRST ? (bitrev(base, a.L - a.k) << a.k) : base;
#pragma unroll
    for (int e = 0; e < E; e++) {
      const unsigned m = m0 | ((unsigned)e << f_prev);
      const unsigned g = FIRST ? obase + m : obase + (m << a.s0);
      Fr y = x[e];
      if (INVERSE && a.last) y = ntt_mul(coset ? fr_load(coset + g) : a.ninv, y);   // reduced factor first: y may be lazy
      else if (a.last) y = bf_out(y);
      fr_store(out + g, y);
    }
  }
}

int ntt_get_twiddles(tp_ctx* ctx, unsigned log_n, const Fr** tw) {
  auto it = ctx->ntt_tables.find(log_n);
  if (it == ctx->ntt_tables.end()) {
    NttTables t;
    size_t count = ((size_t)1 << log_n) / 2 + 1;
    TP_CUDA_OK(ctx, cudaMalloc(&t.tw, count * sizeof(Fr)));
    Fr w = to_dev(omega_for_log(log_n));
    size_t threads = (count + 15) / 16;
    k_pow_table<<<(unsigned)((threads + 127) / 128), 128, 0, ctx->stream>>>(t.tw, w, count, to_dev(tph::HFr::one()));
    TP_LAUNCH(ctx, "k_pow_table");
    it = ctx->ntt_tables.emplace(log_n, t).first;
  }
  *tw = it->second.tw;
  return TP_OK;
}

// scale * g^i for i < 2^log_n (scale = n^-1 for the inverse transform's output table)
static int get_coset_table(tp_ctx* ctx, unsigned log_n, const tph::HFr& g, bool scaled, const Fr** out) {
  for (auto& c : ctx->coset_tables) {
    if (c.log_n == log_n && c.scaled == (scaled ? 1 : 0) && memcmp(c.g, g.v, 32) == 0) {
      *out = c.lo;
      return TP_OK;
    }
  }
  CosetTable c;
  c.log_n = log_n;
  c.scaled = scaled ? 1 : 0;
  memcpy(c.g, g.v, 32);
  size_t n = (size_t)1 << log_n;
  TP_CUDA_OK(ctx, cudaMalloc(&c.lo, n * sizeof(Fr)));
  tph::HFr scale = scaled ? tph::HFr::from_u64((uint64_t)n).inv() : tph::HFr::one();
  k_pow_table<<<(unsigned)(((n + 15) / 16 + 127) / 128), 128, 0, ctx->stream>>>(c.lo, to_dev(g), n, to_dev(scale));
  TP_LAUNCH(ctx, "k_pow_table");
  ctx->coset_tables.push_back(c);
  *out = c.lo;
  return TP_OK;
}

// Pass plan: as few passes as the tile allows (k <= tile_log - 2 with four columns per tile), every pass at least B
// stages.  The first pass has four columns per tile (its rows are far apart: 128-byte runs); later passes with
// fewer stages widen the tile instead (2^(tile_log - k) adjacent columns), so every CTA has 256 threads.
static int ntt_plan(unsigned log_n, unsigned* ks, unsigned tile_log, unsigned B) {
  if (log_n <= tile_log) {
    ks[0] = log_n;
    return 1;
  }
  const unsigned kmax = tile_log - 2;
  int npass = (int)((log_n + kmax - 1) / kmax);
  unsigned left = log_n;
  for (int i = 0; i < npass; i++) {
    unsigned passes_after = (unsigned)(npass - 1 - i);
    unsigned k = left < kmax ? left : kmax;
    if (left - k < B * passes_after) k = left - B * passes_after;  // leave >= B stages for each later pass
    ks[i] = k;
    left -= k;
  }
  return npass;
}

template <int B>
static int ntt_launch(tp_ctx* ctx, const NttPassArgs& a, dim3 grid, unsigned threads, size_t smem, bool inverse) {
  static bool smem_attr[64] = {false};   // per device: the ranks of a device group launch from their own devices
  if (!smem_attr[ctx->device & 63]) {
    const int cap = (int)((2u << NTT_TILE_LOG(B)) * 16u);
    TP_CUDA_OK(ctx, cudaFuncSetAttribute(k_ntt_r8<B, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    TP_CUDA_OK(ctx, cudaFuncSetAttribute(k_ntt_r8<B, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    TP_CUDA_OK(ctx, cudaFuncSetAttribute(k_ntt_r8<B, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    TP_CUDA_OK(ctx, cudaFuncSetAttribute(k_ntt_r8<B, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    smem_attr[ctx->device & 63] = true;
  }
  if (a.first && inverse) k_ntt_r8<B, true, true><<<grid, threads, smem, ctx->stream>>>(a);
  else if (a.first) k_ntt_r8<B, true, false><<<grid, threads, smem, ctx->stream>>>(a);
  else if (inverse) k_ntt_r8<B, false, true><<<grid, threads, smem, ctx->stream>>>(a);
  else k_ntt_r8<B, false, false><<<grid, threads, smem, ctx->stream>>>(a);
  TP_LAUNCH(ctx, "k_ntt_r8");
  return TP_OK;
}

// `count` transforms of size 2^log_n in one set of launches; coset[i] (Montgomery generator, may be
// null) selects the coset of entry i.  in[i] == out[i] is allowed (a scratch copy takes the first pass).
int ntt_batch_dev(tp_ctx* ctx, const Fr* const* in, Fr* const* out, const uint64_t* const* coset, int count,
                  unsigned log_n, bool inverse) {
  if (count <= 0) return TP_OK;
  if (count > NTT_MAX_BATCH) {
    TP_TRY(ntt_batch_dev(ctx, in, out, coset, NTT_MAX_BATCH, log_n, inverse));
    return ntt_batch_dev(ctx, in + NTT_MAX_BATCH, out + NTT_MAX_BATCH, coset ? coset + NTT_MAX_BATCH : nullptr,
                         count - NTT_MAX_BATCH, log_n, inverse);
  }
  if (log_n == 0) {
    for (int i = 0; i < count; i++)
      if (in[i] != out[i]) TP_CUDA_OK(ctx, cudaMemcpyAsync(out[i], in[i], sizeof(Fr), cudaMemcpyDeviceToDevice, ctx->stream));
    return TP_OK;
  }
  if (log_n > 28) return fail(ctx, TP_ERR_INVALID_ARG, "ntt: log_n > 28");
  ProfScope prof(ctx, TP_PHASE_NTT);
  const Fr* tw;
  TP_TRY(ntt_get_twiddles(ctx, log_n, &tw));
  size_t n = (size_t)1 << log_n;
  tph::HFr ninv = tph::HFr::from_u64((uint64_t)n).inv();
  NttPassArgs a;
  a.tw = tw;
  a.L = log_n;
  a.inverse = inverse ? 1 : 0;
  a.ninv = to_dev(ninv);
  for (int i = 0; i < NTT_MAX_BATCH; i++) {
    const int s = i < count ? i : 0;
    a.coset[i] = nullptr;
    if (coset && coset[s]) {
      tph::HFr g;
      memcpy(g.v, coset[s], 32);
      if (inverse) g = g.inv();
      TP_TRY(get_coset_table(ctx, log_n, g, inverse, &a.coset[i]));
    }
  }
  if (log_n < 3) {
    for (int i = 0; i < NTT_MAX_BATCH; i++) {
      a.in[i] = in[i < count ? i : 0];
      a.out[i] = out[i < count ? i : 0];
    }
    a.s0 = 0;
    a.k = log_n;
    a.cw = 0;
    a.first = a.last = 1;
    k_ntt_small<<<dim3(1, (unsigned)count), 32, 0, ctx->stream>>>(a);
    TP_LAUNCH(ctx, "k_ntt_small");
    return TP_OK;
  }
  // elements per thread: 8 (B = 3) or 4 (B = 2); tp_ctx_set_option("ntt_radix_log", 2 | 3) / $TP_NTT_B
  static const char* env_b = getenv("TP_NTT_B");
  const unsigned B = (env_b && (*env_b == '2' || *env_b == '3')) ? (unsigned)(*env_b - '0') : ctx->ntt_radix_log;
  const unsigned tile_log = NTT_TILE_LOG(B);
  unsigned ks[8];
  const int npass = ntt_plan(log_n, ks, tile_log, B);
  // the first pass of a multi-pass transform is out of place: in-place entries go through scratch
  Fr* scratch = nullptr;
  if (npass > 1) {
    int inplace = 0;
    for (int i = 0; i < count; i++) inplace += in[i] == out[i];
    if (inplace) {
      TP_TRY(ensure(ctx, ctx->ntt_scratch, (size_t)inplace * n * sizeof(Fr)));
      scratch = (Fr*)ctx->ntt_scratch.p;
    }
  }
  const Fr* src[NTT_MAX_BATCH];
  for (int i = 0; i < count; i++) src[i] = in[i];
  unsigned s0 = 0;
  for (int p = 0; p < npass; p++) {
    Fr* sc = scratch;
    for (int i = 0; i < NTT_MAX_BATCH; i++) {
      const int s = i < count ? i : 0;
      a.in[i] = src[s];
      a.out[i] = out[s];
      if (i < count && p == 0 && npass > 1 && in[i] == out[i]) {
        a.out[i] = sc;
        sc += n;
      }
    }
    a.s0 = s0;
    a.k = ks[p];
    a.cw = npass == 1 ? 0 : (p == 0 ? 2 : tile_log - a.k);
    a.first = (p == 0);
    a.last = (p == npass - 1);
    const unsigned T = 1u << (a.k + a.cw);
    const unsigned grid = (unsigned)(n >> (a.k + a.cw));
    const dim3 g3(grid, (unsigned)count);
    const size_t smem = 2 * T * sizeof(uint4);
    if (B == 3) TP_TRY(ntt_launch<3>(ctx, a, g3, T >> 3, smem, inverse));
    else TP_TRY(ntt_launch<2>(ctx, a, g3, T >> 2, smem, inverse));
    for (int i = 0; i < count; i++) src[i] = a.out[i];
    s0 += a.k;
  }
  return TP_OK;
}

int ntt_dev(tp_ctx* ctx, const Fr* in, Fr* out, unsigned log_n, bool inverse, const uint64_t* coset) {
  const Fr* ins[1] = {in};
  Fr* outs[1] = {out};
  const uint64_t* cos[1] = {coset};
  return ntt_batch_dev(ctx, ins, outs, cos, 1, log_n, inverse);
}

}  // namespace tp
