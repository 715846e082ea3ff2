// KZG commit as a Pippenger G1 multi-scalar multiplication for sm_100a.
//
// Replaces `KzgScheme::evaluate_in_s` (kzg/src/lib.rs:41-54), which the reference computes as
// n independent double-and-add scalar multiplications folded with `Sum`.  The affine result of
// a group sum is unique, so the bucket method is bit-exact with it.
//
// Stages (in order on the ctx stream; the opt-in "pipeline" mode near the end of this file spreads the stages of
// consecutive sub-batches over three streams instead):
//   1. k_msm_digits   : scalar Montgomery -> canonical, signed-digit windows of c bits; each
//                       non-zero digit takes a rank in its bucket with one atomicAdd
//                       (histogram and within-bucket rank in a single pass)
//   2. k_scan_*       : exclusive scan of the bucket histogram -> bucket offsets
//   3. k_msm_scatter  : counting-sort scatter of (point index | sign) and bucket key
//   4. k_msm_accumulate: load-balanced segmented accumulation -- every thread owns a fixed-size
//                       chunk of the sorted entries (not a bucket), adds SRS points in XYZZ mixed
//                       coordinates, writes complete runs straight to their bucket and emits
//                       head/tail partials for runs that cross chunk boundaries
//   5. k_msm_merge    : stitches the boundary partials
//   6. k_msm_wsum_level / k_msm_rowcol / k_msm_bitsums: sum_v v * B_v of each bucket set without a
//                       single scalar multiplication: (big sets) one level of 16-bucket running sums,
//                       then row / column tree sums, then the remaining index bits as masked tree
//                       sums (see "bucket reduction" below)
//   7. sharded over GPUs (comm.cu): every rank does 1-6 for the buckets it owns; the ranks' step-6
//                       outputs are all-gathered on the stream and combined by k_msm_combine
//   8. host           : ~50 additions/doublings per bucket set + affine conversion (serial tail;
//                       one CPU thread is ~10x faster than one GPU thread at 381-bit arithmetic).
//
// Fixed-base tables: the SRS never changes, so tp_srs holds `levels` copies of it, level k =
// 2^(c k) * P_i (srs.cu).  Window w of scalar i then adds table[w % levels][i] into bucket set
// w / levels, i.e. with levels == nwin ALL windows of an MSM share ONE set of 2^(c-1) buckets: the
// bucket reduction shrinks nwin-fold, which in turn lets c grow (fewer windows = fewer additions).
#include <stdlib.h>

#include <utility>

#include "common.cuh"

#include <future>
#include <system_error>

namespace tp {

#define MSM_NONE 0x7fffffffu
#define MSM_IDENT 0x80000000u   // partial slot holds the identity (point not stored)

// Tunables (defaults chosen on B200; TP_MSM_CHUNK / TP_MSM_C / TP_MSM_LEVELS override for sweeps).
static unsigned env_uint(const char* name, unsigned dflt) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  long x = strtol(v, nullptr, 10);
  return x > 0 ? (unsigned)x : dflt;
}
static bool msm_force_levels() { static unsigned v = env_uint("TP_MSM_FORCE_LEVEL_MERGE", 0); return v != 0; }
static unsigned msm_chunk() { static unsigned v = env_uint("TP_MSM_CHUNK", 64); return v; }   // sorted entries per accumulate thread

struct MsmPlan {
  unsigned c;        // window bits
  unsigned nwin;     // number of windows
  unsigned nbuck;    // buckets per set THIS RANK owns: 2^(c-1) on one GPU; sharded, rank r of `world` owns the global
                     // buckets b with b % world == r as local bucket b / world (count rounded up to a power of two)
  unsigned levels;   // fixed-base table levels held by the SRS
  unsigned nsets;    // bucket sets per MSM = ceil(nwin / levels)
};

static unsigned windows_for(unsigned c) {
  unsigned nwin = (255 + c - 1) / c;
  unsigned top_bits = 255 - (nwin - 1) * c;
  if (top_bits == c) nwin++;  // signed carry out of a full top window
  return nwin;
}

// Window size and table depth for an SRS of `table_len` points of which one MSM call touches `len`, when `budget`
// bytes may go to tables.  Cost in Fq multiplications: 10 per bucket addition (XYZZ mixed), ~30 per bucket in the
// reduction; sharded over `world` ranks by bucket, both terms shrink 1/world, so the plan is that of one GPU.
void msm_choose_tables(size_t len, size_t table_len, size_t budget, unsigned world, unsigned* c_out, unsigned* levels_out) {
  static unsigned force_c = env_uint("TP_MSM_C", 0);
  static unsigned max_levels = env_uint("TP_MSM_LEVELS", 1u << 30);
  double best_cost = 1e300;
  unsigned best_c = 2, best_l = 1;
  size_t n = len ? len : 1;
  size_t tn = table_len ? table_len : 1;
  size_t afford = budget / (tn * sizeof(G1Affine));
  if (afford < 1) afford = 1;
  for (unsigned c = 2; c <= 26; c++) {
    if (force_c && c != force_c) continue;
    unsigned nwin = windows_for(c);
    unsigned levels = nwin;
    if (levels > afford) levels = (unsigned)afford;
    if (levels > max_levels) levels = max_levels;
    if ((size_t)levels * tn >= ((size_t)1 << 31)) levels = (unsigned)((((size_t)1 << 31) - 1) / tn);
    if (levels < 1) levels = 1;
    unsigned nsets = (nwin + levels - 1) / levels;
    levels = (nwin + nsets - 1) / nsets;  // no deeper than the set count needs
    double nb = (double)(1u << (c - 1));
    const double w = world ? (double)world : 1.0;
    double cost = (double)n * nwin * 10.0 / w + nsets * nb * 30.0 / w + nsets * 3000.0;
    unsigned top_bits = 255 - (nwin - 1) * c;
    if (levels == 1 && top_bits + 6 < c && n > 4096) cost += 25e6;  // a lone top window funnels ~n points into few buckets
    if (cost < best_cost) {
      best_cost = cost;
      best_c = c;
      best_l = levels;
    }
  }
  *c_out = best_c;
  *levels_out = best_l;
}

static MsmPlan msm_plan(const tp_srs* srs, unsigned world) {
  MsmPlan pl;
  pl.c = srs->c;
  pl.nwin = windows_for(pl.c);
  pl.nbuck = 1u << (pl.c - 1);
  if (world > 1) {
    const unsigned need = (pl.nbuck + world - 1) / world;
    unsigned p2 = 1;
    while (p2 < need) p2 <<= 1;
    pl.nbuck = p2;
  }
  pl.levels = srs->levels;
  pl.nsets = (pl.nwin + pl.levels - 1) / pl.levels;
  return pl;
}

// ---- 1. digits + histogram/rank ----------------------------------------------------------
#define MSM_MAX_BATCH 16
struct MsmScalarSets {
  const Fr* p[MSM_MAX_BATCH];
};
// blockIdx.y = batch element b.  Window w goes to bucket set b * nsets + w / levels; the entry
// arrays stay window-major ((b * nwin + w) * n + i) so the scatter can recover (w, i).
// Sharded (world > 1): every rank walks all scalars, but only the digits whose bucket it owns
// (bucket % world == my_rank) take a histogram slot; the others leave MSM_NONE in the key array and cost one coalesced 4-byte store.
__global__ void k_msm_digits(MsmScalarSets sets, size_t n, unsigned c, unsigned nwin, unsigned nbuck, unsigned levels,
                             unsigned nsets, unsigned world, unsigned my_rank, unsigned* __restrict__ hist,
                             unsigned* __restrict__ keys, unsigned* __restrict__ ranks) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned wbase = blockIdx.y * nwin;
  const unsigned sbase = blockIdx.y * nsets;
  Fr s = fr_from_mont(fr_load(sets.p[blockIdx.y] + i));
  unsigned carry = 0;
  for (unsigned w = 0; w < nwin; w++) {
    unsigned bit = w * c;
    unsigned raw = 0;
    if (bit < 256) {
      unsigned limb = bit >> 5, off = bit & 31;
      unsigned long long two = s.v[limb];
      if (limb + 1 < 8) two |= (unsigned long long)s.v[limb + 1] << 32;
      raw = (unsigned)(two >> off) & ((1u << c) - 1);
    }
    raw += carry;
    unsigned key = MSM_NONE, rank = 0;   // rank = position of the entry inside its bucket
    carry = 0;
    if (raw != 0) {
      unsigned mag = raw, neg = 0;
      if (raw > (1u << (c - 1))) {
        mag = (1u << c) - raw;
        neg = 1;
        carry = 1;
      }
      if (mag != 0) {
        unsigned b = mag - 1;
        bool mine = true;
        if (world > 1) {
          mine = (b % world) == my_rank;
          b /= world;
        }
        if (mine) {
          unsigned k = (sbase + w / levels) * nbuck + b;
          rank = atomicAdd(&hist[k], 1u);
          key = k | (neg << 31);
        }
      }
    }
    keys[(size_t)(wbase + w) * n + i] = key;
    if (key != MSM_NONE) ranks[(size_t)(wbase + w) * n + i] = rank;   // the scatter reads ranks of owned entries only
  }
}

// ---- 1b. digits of a sharded MSM ----------------------------------------------------------------
// Rank r of `world` owns the buckets b with b % world == r.  Every rank walks ALL scalars (digit extraction is cheap)
// but only about 1 / world of the digits are its own: writing a window-major key array for all of them and reading it
// back in the scatter would cost every rank the memory traffic of an unsharded MSM.  Instead the owned entries go to a
// COMPACT list -- (bucket key | sign, rank inside the bucket, table index) -- in blocks: a thread first computes its
// digits and takes their histogram slots, the block sums its threads' counts and reserves its share of the list with one
// atomicAdd, and the threads write their entries there.  The scatter then runs over the compact list only.
struct MsmEntry {
  unsigned key, rank, idx;
};
#define MSM_MAX_WIN 128   // windows_for(2) = 128
// c-bit field w of the canonical scalar (no carry applied)
__device__ __forceinline__ unsigned msm_raw_digit(const Fr& s, unsigned w, unsigned c) {
  const unsigned bit = w * c;
  if (bit >= 256) return 0;
  const unsigned limb = bit >> 5, off = bit & 31;
  unsigned long long two = s.v[limb];
  if (limb + 1 < 8) two |= (unsigned long long)s.v[limb + 1] << 32;
  return (unsigned)(two >> off) & ((1u << c) - 1);
}
// Ownership of bucket b: rank b % world, local index b / world -- a mask and a shift when world is a power of two (the
// general division costs more than the digit extraction itself, and every rank pays it for ALL digits).
struct MsmOwner {
  unsigned world, rank, mask, shift;   // shift == 32: world is not a power of two
  __device__ __forceinline__ bool mine(unsigned b) const { return shift != 32 ? (b & mask) == rank : b % world == rank; }
  __device__ __forceinline__ unsigned local(unsigned b) const { return shift != 32 ? b >> shift : b / world; }
};
__global__ void __launch_bounds__(256) k_msm_digits_sharded(MsmScalarSets sets, size_t n, unsigned c, unsigned nwin, unsigned nbuck,
                                                            unsigned levels, unsigned nsets, MsmOwner own,
                                                            unsigned stride, unsigned* __restrict__ hist,
                                                            unsigned* __restrict__ list_count, MsmEntry* __restrict__ list) {
  __shared__ unsigned warp_tot[8];
  __shared__ unsigned block_base;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned sbase = blockIdx.y * nsets;
  Fr s;
  if (i < n) s = fr_from_mont(fr_load(sets.p[blockIdx.y] + i));
  const unsigned half = 1u << (c - 1);
  // pass 1: one walk over the windows notes which digits are this rank's and the carry that entered each of them (a bit
  // each: nwin <= 32, i.e. c >= 8); pass 2 visits the owned windows only -- about nwin / world of them
  unsigned own_mask = 0, carry_mask = 0, mine = 0;
  const bool masks = nwin <= 32;
  auto walk = [&](auto&& emit) {
    unsigned carry = 0;
    for (unsigned w = 0; w < nwin; w++) {
      const unsigned raw = msm_raw_digit(s, w, c) + carry;
      const unsigned cin = carry;
      carry = raw > half ? 1u : 0u;
      if (raw == 0 || raw == (1u << c)) continue;
      const unsigned mag = carry ? (1u << c) - raw : raw;
      if (!own.mine(mag - 1)) continue;
      emit(w, cin);
    }
  };
  if (i < n)
    walk([&](unsigned w, unsigned cin) {
      mine++;
      if (masks) {
        own_mask |= 1u << w;
        carry_mask |= cin << w;
      }
    });
  // block-wide exclusive prefix of `mine`
  const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned incl = mine;
  for (unsigned d = 1; d < 32; d <<= 1) {
    unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += v;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (unsigned k = 0; k < blockDim.x / 32; k++) {
      unsigned v = warp_tot[k];
      warp_tot[k] = run;
      run += v;
    }
    block_base = run ? atomicAdd(list_count, run) : 0;
  }
  __syncthreads();
  unsigned pos = block_base + warp_tot[wid] + incl - mine;
  auto put = [&](unsigned w, unsigned cin) {
    const unsigned raw = msm_raw_digit(s, w, c) + cin;
    const unsigned neg = raw > half ? 1u : 0u;
    const unsigned mag = neg ? (1u << c) - raw : raw;
    const unsigned k = (sbase + w / levels) * nbuck + own.local(mag - 1);
    MsmEntry e;
    e.key = k | (neg << 31);
    e.rank = atomicAdd(&hist[k], 1u);
    e.idx = (w % levels) * stride + (unsigned)i;   // level (w % levels) of the fixed-base table holds 2^(c (w % levels)) * P_i
    list[pos++] = e;
  };
  if (i >= n) return;
  if (masks) {
    while (own_mask) {
      const unsigned w = __ffs(own_mask) - 1;
      own_mask &= own_mask - 1;
      put(w, (carry_mask >> w) & 1u);
    }
  } else {
    walk(put);
  }
}
__global__ void __launch_bounds__(256) k_msm_scatter_compact(const MsmEntry* __restrict__ list, const unsigned* __restrict__ count_ptr,
                                                             const unsigned* __restrict__ offsets, uint2* __restrict__ sorted) {
  const unsigned count = *count_ptr;
  for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
    const MsmEntry en = list[e];
    const unsigned k = en.key & MSM_NONE;
    sorted[offsets[k] + en.rank] = make_uint2(en.idx | (en.key & 0x80000000u), k);
  }
}

// ---- 2. exclusive scan (3 kernels; T = u32, or u64 carrying two packed u32 counters) -------------
#define SCAN_BLOCK 1024
template <typename T>
__global__ void k_scan_local(const T* __restrict__ in, T* __restrict__ out, T* __restrict__ sums, size_t n,
                             unsigned* __restrict__ max_out) {
  __shared__ T s[SCAN_BLOCK];
  size_t g = (size_t)blockIdx.x * SCAN_BLOCK + threadIdx.x;
  T v = g < n ? in[g] : 0;
  if (max_out) {  // largest bucket (decides whether chunks can consist of a single run); u32 only
    unsigned wmax = __reduce_max_sync(0xffffffffu, (unsigned)v);
    if ((threadIdx.x & 31) == 0 && wmax > 0) atomicMax(max_out, wmax);
  }
  s[threadIdx.x] = v;
  __syncthreads();
  for (unsigned d = 1; d < SCAN_BLOCK; d <<= 1) {
    T t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
    __syncthreads();
    s[threadIdx.x] += t;
    __syncthreads();
  }
  if (g < n) out[g] = s[threadIdx.x] - v;
  if (threadIdx.x == SCAN_BLOCK - 1) sums[blockIdx.x] = s[threadIdx.x];
}
template <typename T>
__global__ void k_scan_sums(T* sums, size_t nblocks) {
  // single block, serial over tiles of SCAN_BLOCK
  __shared__ T s[SCAN_BLOCK];
  __shared__ T carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (size_t base = 0; base < nblocks; base += SCAN_BLOCK) {
    size_t g = base + threadIdx.x;
    T v = g < nblocks ? sums[g] : 0;
    s[threadIdx.x] = v;
    __syncthreads();
    for (unsigned d = 1; d < SCAN_BLOCK; d <<= 1) {
      T t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
      __syncthreads();
      s[threadIdx.x] += t;
      __syncthreads();
    }
    if (g < nblocks) sums[g] = s[threadIdx.x] - v + carry;
    __syncthreads();
    if (threadIdx.x == SCAN_BLOCK - 1) carry += s[threadIdx.x];
    __syncthreads();
  }
}
template <typename T>
__global__ void k_scan_add(T* out, const T* sums, size_t n) {
  size_t g = (size_t)blockIdx.x * SCAN_BLOCK + threadIdx.x;
  if (g < n) out[g] += sums[blockIdx.x];
}

// ---- 3. scatter ----------------------------------------------------------------------------
// The 8-byte stores of the counting sort land at random positions of one MSM's bucket-sorted list (len * nwin * 8
// bytes: 109 MB at 2^20, as large as the L2), and a store that misses L2 costs DRAM a 32-byte sector read and a
// write-back.  The scatter therefore runs once per SLICE of the bucket range: the stores of a launch fall into a
// region that stays in L2 until its sectors are complete, and the entry arrays being MSM-major keeps that region to
// one MSM at a time.  A launch re-reads every key (4 bytes, four per thread) but touches ranks, offsets and the
// output only for the keys of its slice.  B200, 2^20, 13 MSMs per proof, sort phase: 1 slice 5.8 ms, 2 slices 4.7 ms,
// 4 slices 5.0 ms, 8 slices 7.0 ms (profiles/r1_summary.md Q).
__device__ __forceinline__ void msm_scatter_one(unsigned key, size_t e, const unsigned* __restrict__ ranks,
                                                const unsigned* __restrict__ offsets, size_t n, unsigned nwin,
                                                unsigned levels, unsigned stride, uint2* __restrict__ sorted,
                                                unsigned slice_mask, unsigned slice_shift, unsigned slice) {
  if ((key & MSM_NONE) == MSM_NONE) return;
  const unsigned k = key & MSM_NONE;
  if (((k & slice_mask) >> slice_shift) != slice) return;
  const unsigned pos = offsets[k] + ranks[e];
  const unsigned i = (unsigned)(e % n);
  const unsigned w = (unsigned)(e / n) % nwin;
  // index into the fixed-base table: level (w % levels) holds 2^(c (w % levels)) * P_i
  sorted[pos] = make_uint2(((w % levels) * stride + i) | (key & 0x80000000u), k);  // one 8-byte store
}
#define SCATTER_UNROLL 1
__global__ void __launch_bounds__(256) k_msm_scatter(const unsigned* __restrict__ keys, const unsigned* __restrict__ ranks,
                                                     const unsigned* __restrict__ offsets, size_t n, size_t total,
                                                     unsigned nwin, unsigned levels, unsigned stride,
                                                     uint2* __restrict__ sorted, unsigned slice_mask, unsigned slice_shift,
                                                     unsigned slice) {
  // SCATTER_UNROLL coalesced 16-byte key loads per thread, all issued before any of them is used
  uint4 kk[SCATTER_UNROLL];
  size_t e0[SCATTER_UNROLL];
#pragma unroll
  for (int j = 0; j < SCATTER_UNROLL; j++) {
    e0[j] = (((size_t)blockIdx.x * SCATTER_UNROLL + j) * blockDim.x + threadIdx.x) * 4;
    kk[j] = make_uint4(MSM_NONE, MSM_NONE, MSM_NONE, MSM_NONE);
    if (e0[j] + 4 <= total) {   // the key array is 16-byte aligned: cudaMalloc'ed, e0 a multiple of 4
      kk[j] = *reinterpret_cast<const uint4*>(keys + e0[j]);
    } else if (e0[j] < total) {
      kk[j].x = keys[e0[j]];
      if (e0[j] + 1 < total) kk[j].y = keys[e0[j] + 1];
      if (e0[j] + 2 < total) kk[j].z = keys[e0[j] + 2];
    }
  }
#pragma unroll
  for (int j = 0; j < SCATTER_UNROLL; j++) {
    msm_scatter_one(kk[j].x, e0[j], ranks, offsets, n, nwin, levels, stride, sorted, slice_mask, slice_shift, slice);
    msm_scatter_one(kk[j].y, e0[j] + 1, ranks, offsets, n, nwin, levels, stride, sorted, slice_mask, slice_shift, slice);
    msm_scatter_one(kk[j].z, e0[j] + 2, ranks, offsets, n, nwin, levels, stride, sorted, slice_mask, slice_shift, slice);
    msm_scatter_one(kk[j].w, e0[j] + 3, ranks, offsets, n, nwin, levels, stride, sorted, slice_mask, slice_shift, slice);
  }
}

// ---- 4a. batch-affine rounds --------------------------------------------------------------
// Before the XYZZ accumulation the bucket-sorted entry list is halved a few times in AFFINE
// coordinates: in every round each bucket pairs its entries (2q, 2q+1) and replaces a pair by its
// sum, an odd last entry passes through.  An affine addition is 1 inversion + 2M + 1S; the
// inversion is shared by the AFF_K pairs one thread owns (Montgomery's trick: 3M per pair) and is
// itself done by division steps on the ALU pipe (fq_inv.cuh), so a pair costs 5M + 1S = 1662 wide
// multiplies against 2604 for the XYZZ mixed addition -- the FMA-heavy pipe is what bounds the MSM.
// Work is assigned by PAIR index (a scan of pairs per bucket), so every lane of a warp has exactly
// AFF_K real additions whatever the bucket sizes are.
//
// Points are addressed through one index space: idx < split -> fixed-base table, else -> scratch
// array of sums (round outputs); entries that pass through unpaired keep their index (and sign).
#define AFF_K 32            // most pairs per thread (local array of prefix products)
#define AFF_MAX_ROUNDS 8
__device__ __forceinline__ const G1Affine* msm_point(const G1Affine* __restrict__ bases, const G1Affine* __restrict__ scratch,
                                                     unsigned split, unsigned idx31) {
  return idx31 < split ? bases + idx31 : scratch + (idx31 - split);
}
__device__ __forceinline__ G1Affine msm_point_load(const G1Affine* __restrict__ bases, const G1Affine* __restrict__ scratch,
                                                   unsigned split, unsigned idx) {
  G1Affine p = affine_load(msm_point(bases, scratch, split, idx & 0x7fffffffu));
  if (idx >> 31) p.y = fq_neg(p.y);
  return p;
}

// per bucket: pairs this round and entries next round, packed as (next << 32 | pairs) for ONE scan
__global__ void k_aff_plan(const unsigned* __restrict__ cnt_in, size_t nkeys, unsigned* __restrict__ cnt_out,
                           unsigned long long* __restrict__ packed) {
  size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nkeys) return;
  unsigned c = b < nkeys ? cnt_in[b] : 0;
  unsigned nxt = (c + 1) >> 1;
  if (b < nkeys) cnt_out[b] = nxt;
  packed[b] = ((unsigned long long)nxt << 32) | (c >> 1);
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem));
}

// One thread per entry of the round's input list: the even entries of a bucket open a pair and
// write its record (index | sign of both operands, output position, bucket) at the pair's global
// index, an odd last entry passes through to the next list.  No searching: an entry carries its
// bucket, the scanned plan gives the bucket's first pair and its first output slot.
__global__ void k_aff_records(const uint2* __restrict__ l_in, const unsigned* __restrict__ m_ptr,
                              const unsigned* __restrict__ cnt_in, const unsigned* __restrict__ off_in, unsigned off_stride,
                              const unsigned long long* __restrict__ plan, uint4* __restrict__ rec,
                              uint2* __restrict__ l_out) {
  const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= *m_ptr) return;
  const uint2 ent = l_in[e];
  const unsigned b = ent.y;
  const unsigned q = e - off_in[(size_t)b * off_stride];
  if (q & 1) return;
  const unsigned long long pl = plan[b];
  const unsigned o = (unsigned)(pl >> 32) + (q >> 1);
  if (q + 1 < cnt_in[b]) {
    rec[(unsigned)pl + (q >> 1)] = make_uint4(ent.x, l_in[e + 1].x, o, b);
  } else {
    l_out[o] = ent;
  }
}

// AFF_THREADS threads share ONE inversion: every thread multiplies up the denominators of its
// k_run pairs, the block multiplies the thread products together (prefix and suffix scans in
// shared memory), warp 0 inverts the block product by division steps, and every thread gets its
// own inverse back with two more multiplications.
#define AFF_THREADS 128
#define AFF_SMEM_STAGE (2 * 12 * AFF_THREADS * 16)              // cp.async staging: [2 stages][12 chunks][thread] x 16 B
#define AFF_SMEM (AFF_SMEM_STAGE)                                // the scans reuse the staging area
__device__ __forceinline__ Fq sh_fq_load(const uint32_t* base, unsigned t) {  // limb-major: conflict-free
  Fq r;
#pragma unroll
  for (int i = 0; i < 12; i++) r.v[i] = base[i * AFF_THREADS + t];
  return r;
}
__device__ __forceinline__ void sh_fq_store(uint32_t* base, unsigned t, const Fq& a) {
#pragma unroll
  for (int i = 0; i < 12; i++) base[i * AFF_THREADS + t] = a.v[i];
}

__global__ void __launch_bounds__(AFF_THREADS, 4) k_aff_round(const G1Affine* __restrict__ bases, G1Affine* __restrict__ scratch,
                                                              unsigned split, const uint4* __restrict__ rec,
                                                              const unsigned long long* __restrict__ plan, unsigned nkeys,
                                                              uint2* __restrict__ l_out, unsigned region, unsigned k_run) {
  extern __shared__ uint4 aff_sh[];
  const unsigned pairs_total = (unsigned)plan[nkeys];
  const unsigned block_p0 = blockIdx.x * AFF_THREADS * k_run;
  if (block_p0 >= pairs_total) return;  // whole block idle (grid sized from an upper bound)
  const unsigned p0 = block_p0 + threadIdx.x * k_run;
  const unsigned np = p0 >= pairs_total ? 0 : (pairs_total - p0 < k_run ? pairs_total - p0 : k_run);
  const uint4* my = rec + p0;
  Fq pre[AFF_K];
  // Operands travel global -> shared with cp.async one pair ahead of the arithmetic (thread-private
  // slots, chunk-major so that a warp's 16-byte accesses are conflict-free).
  auto stage_pair = [&](int stage, const uint4& rc, int chunks_per_point) {
    const uint4* a1 = (const uint4*)msm_point(bases, scratch, split, rc.x & 0x7fffffffu);
    const uint4* a2 = (const uint4*)msm_point(bases, scratch, split, rc.y & 0x7fffffffu);
    for (int c = 0; c < chunks_per_point; c++) {
      cp_async16(&aff_sh[(stage * 12 + c) * AFF_THREADS + threadIdx.x], a1 + c);
      cp_async16(&aff_sh[(stage * 12 + 6 + c) * AFF_THREADS + threadIdx.x], a2 + c);
    }
    asm volatile("cp.async.commit_group;");
  };
  auto staged_fq = [&](int stage, int chunk0) {
    Fq r;
    const uint4 a = aff_sh[(stage * 12 + chunk0) * AFF_THREADS + threadIdx.x],
                b = aff_sh[(stage * 12 + chunk0 + 1) * AFF_THREADS + threadIdx.x],
                c = aff_sh[(stage * 12 + chunk0 + 2) * AFF_THREADS + threadIdx.x];
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    r.v[8] = c.x; r.v[9] = c.y; r.v[10] = c.z; r.v[11] = c.w;
    return r;
  };
  Fq acc = fq_one();
  uint4 rc_next = np ? my[0] : make_uint4(0, 0, 0, 0);
  uint4 rc_next2 = np > 1 ? my[1] : rc_next;   // records run two pairs ahead, operands one pair ahead
  if (np) stage_pair(0, rc_next, 3);
  for (unsigned i = 0; i < np; i++) {
    const uint4 rc = rc_next;
    if (i + 1 < np) {
      rc_next = rc_next2;
      if (i + 2 < np) rc_next2 = my[i + 2];
      stage_pair((i + 1) & 1, rc_next, 3);
      asm volatile("cp.async.wait_group 1;");
    } else {
      asm volatile("cp.async.wait_group 0;");
    }
    const Fq x1 = staged_fq(i & 1, 0), x2 = staged_fq(i & 1, 6);
    Fq d = fq_sub(x2, x1);
    if (fq_is_zero(d) || fq_is_zero(x1) || fq_is_zero(x2)) {  // doubling, cancellation or an identity operand
      G1Affine f1 = msm_point_load(bases, scratch, split, rc.x), f2 = msm_point_load(bases, scratch, split, rc.y);
      Fq ds;
      affine_pair_special(f1, f2, ds);
      d = ds;
    }
    pre[i] = acc;
    acc = fq_mul(acc, d);
  }
  // ---- block-wide inversion of the thread products ----
  __syncthreads();  // staging area is free
  uint32_t* pa = (uint32_t*)aff_sh;                       // inclusive prefix products
  uint32_t* sa = pa + 12 * AFF_THREADS;                   // inclusive suffix products
  uint32_t* tot = sa + 12 * AFF_THREADS;                  // inverse of the block product
  const unsigned t = threadIdx.x;
  sh_fq_store(pa, t, acc);
  sh_fq_store(sa, t, acc);
  __syncthreads();
  for (unsigned dlt = 1; dlt < AFF_THREADS; dlt <<= 1) {
    Fq vp, vs;
    const bool hp = t >= dlt, hs = t + dlt < AFF_THREADS;
    if (hp) vp = fq_mul(sh_fq_load(pa, t), sh_fq_load(pa, t - dlt));
    if (hs) vs = fq_mul(sh_fq_load(sa, t), sh_fq_load(sa, t + dlt));
    __syncthreads();
    if (hp) sh_fq_store(pa, t, vp);
    if (hs) sh_fq_store(sa, t, vs);
    __syncthreads();
  }
  if (t < 32) {
    Fq all = sh_fq_load(pa, AFF_THREADS - 1);
    Fq iv = fq_inverse(all);
    if (t == 0) {
#pragma unroll
      for (int i = 0; i < 12; i++) tot[i] = iv.v[i];
    }
  }
  __syncthreads();
  Fq inv;
#pragma unroll
  for (int i = 0; i < 12; i++) inv.v[i] = tot[i];
  if (t > 0) inv = fq_mul(inv, sh_fq_load(pa, t - 1));
  if (t + 1 < AFF_THREADS) inv = fq_mul(inv, sh_fq_load(sa, t + 1));
  __syncthreads();  // scans done: the area goes back to staging
  // ---- backward: one addition per pair ----
  if (np) {
    rc_next = my[np - 1];
    rc_next2 = np > 1 ? my[np - 2] : rc_next;
    stage_pair((np - 1) & 1, rc_next, 6);
  }
  for (int i = (int)np - 1; i >= 0; i--) {
    const uint4 rc = rc_next;
    if (i > 0) {
      rc_next = rc_next2;
      if (i > 1) rc_next2 = my[i - 2];
      stage_pair((i - 1) & 1, rc_next, 6);
      asm volatile("cp.async.wait_group 1;");
    } else {
      asm volatile("cp.async.wait_group 0;");
    }
    G1Affine p1, p2;
    p1.x = staged_fq(i & 1, 0);
    p1.y = staged_fq(i & 1, 3);
    p2.x = staged_fq(i & 1, 6);
    p2.y = staged_fq(i & 1, 9);
    if (rc.x >> 31) p1.y = fq_neg(p1.y);
    if (rc.y >> 31) p2.y = fq_neg(p2.y);
    Fq d = fq_sub(p2.x, p1.x);
    int kind = 0;
    if (fq_is_zero(d) || fq_is_zero(p1.x) || fq_is_zero(p2.x)) {
      G1Affine f1 = p1, f2 = p2;  // copies: the hot operands never have their address taken
      Fq ds;
      kind = affine_pair_special(f1, f2, ds);
      d = ds;
    }
    const Fq dinv = fq_mul(inv, pre[i]);
    inv = fq_mul(inv, d);
    const G1Affine r = affine_pair_finish(p1, p2, kind, dinv);
    G1Affine* dst = scratch + region + rc.z;
    fq_store(&dst->x, r.x);
    fq_store(&dst->y, r.y);
    l_out[rc.z] = make_uint2(split + region + rc.z, rc.w);
  }
}

// ---- 4b. segmented accumulation --------------------------------------------------------------
// part_keys[2t], part_keys[2t+1]: keys of the head / tail partial of chunk t (MSM_NONE if absent)
#ifndef TP_ACC_MIN_BLOCKS
#define TP_ACC_MIN_BLOCKS 3   // 162 registers, 3 warps per scheduler: FMA-heavy pipe 80 % -> 87 % busy (profiles N)
#endif
// STAGED: the table point of entry e + 1 travels global -> shared memory with cp.async (a thread-private 96-byte slot, two
// stages) while the addition of entry e runs, instead of stalling the addition on a load from a multi-GB table with
// three warps per scheduler to cover it; costs no registers (a prefetch hint into L1 / L2 measured slower, section 7 of
// DESIGN.md).
// LAZY (option msm_fq_lazy, default on): the XYZZ laws on Fq values in [0, 2q) (ec.cuh FqOps<true>) in this kernel and in
// every later one of the MSM -- buckets, partials and running sums are stored lazy -- until the reduction's outputs are
// normalised to [0, q) in k_msm_treesum / k_msm_combine.  The same points mod q as the canonical laws, so the same bytes.
#define ACC_THREADS 128
template <bool STAGED, bool LAZY>
__global__ void __launch_bounds__(ACC_THREADS, TP_ACC_MIN_BLOCKS) k_msm_accumulate(const G1Affine* __restrict__ bases,
                                                        const G1Affine* __restrict__ scratch, unsigned split,
                                                        const uint2* __restrict__ sorted /* (index | sign, key) */,
                                                        const unsigned* __restrict__ m_ptr /* live entry count */,
                                                        unsigned nchunks,
                                                        G1Xyzz* __restrict__ buckets, unsigned* __restrict__ part_keys,
                                                        G1Xyzz* __restrict__ part_pts, unsigned chunk) {
  __shared__ uint4 stage_sh[STAGED ? 2 * 6 * ACC_THREADS : 1];   // [stage][16-byte piece][thread]: conflict-free
  unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nchunks) return;
  const unsigned m_total = *m_ptr;
  unsigned start = t * chunk;
  if (start >= m_total) {  // the grid is sized from an upper bound of the list length
    part_keys[2 * t] = MSM_NONE | MSM_IDENT;
    part_keys[2 * t + 1] = MSM_NONE | MSM_IDENT;
    return;
  }
  unsigned end = start + chunk < m_total ? start + chunk : m_total;
  G1Xyzz acc = xyzz_identity();
  unsigned cur = sorted[start].y;
  bool is_first_run = true;
  auto stage_point = [&](unsigned st, unsigned idx) {
    const uint4* src = (const uint4*)msm_point(bases, scratch, split, idx & 0x7fffffffu);
#pragma unroll
    for (int c = 0; c < 6; c++) cp_async16(&stage_sh[(st * 6 + c) * ACC_THREADS + threadIdx.x], src + c);
    asm volatile("cp.async.commit_group;");
  };
  uint2 ent_next = sorted[start];
  if (STAGED) stage_point(0, ent_next.x);
  for (unsigned e = start; e < end; e++) {
    const uint2 ent = STAGED ? ent_next : sorted[e];
    if (STAGED) {
      if (e + 1 < end) {
        ent_next = sorted[e + 1];
        stage_point((e + 1 - start) & 1, ent_next.x);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
    }
    const unsigned key = ent.y;
    if (key != cur) {
      if (is_first_run) {
        part_keys[2 * t] = cur;
        xyzz_store(part_pts + 2 * t, acc);
        is_first_run = false;
      } else {
        xyzz_store(buckets + cur, acc);  // complete interior run: exclusive owner of the bucket
      }
      acc = xyzz_identity();
      cur = key;
    }
    const unsigned idx = ent.x;
    G1Affine p;
    if (STAGED) {
      const unsigned st = (e - start) & 1;
      uint4 w[6];
#pragma unroll
      for (int c = 0; c < 6; c++) w[c] = stage_sh[(st * 6 + c) * ACC_THREADS + threadIdx.x];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        p.x.v[4 * c] = w[c].x; p.x.v[4 * c + 1] = w[c].y; p.x.v[4 * c + 2] = w[c].z; p.x.v[4 * c + 3] = w[c].w;
        p.y.v[4 * c] = w[3 + c].x; p.y.v[4 * c + 1] = w[3 + c].y; p.y.v[4 * c + 2] = w[3 + c].z; p.y.v[4 * c + 3] = w[3 + c].w;
      }
    } else {
#ifdef TP_ACC_PREFETCH
      // The next entry's point sits anywhere in a multi-GB table: ask for its line(s) now, one addition
      // (thousands of cycles) ahead of the load, instead of stalling on an HBM miss with three warps per scheduler.
      if (e + 1 < end) {
        const char* nx = (const char*)msm_point(bases, scratch, split, sorted[e + 1].x & 0x7fffffffu);
#if TP_ACC_PREFETCH == 2
        asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + 80));
#else
        asm volatile("prefetch.global.L1 [%0];" ::"l"(nx));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(nx + 80));
#endif
      }
#endif
      p = affine_load(msm_point(bases, scratch, split, idx & 0x7fffffffu));
    }
    if (!affine_is_identity(p)) xyzz_madd<LAZY>(acc, p, (idx >> 31) != 0);
  }
  if (is_first_run) {
    part_keys[2 * t] = cur;
    xyzz_store(part_pts + 2 * t, acc);
    part_keys[2 * t + 1] = cur | MSM_IDENT;  // single-run chunk: empty tail partial
  } else {
    part_keys[2 * t + 1] = cur;
    xyzz_store(part_pts + 2 * t + 1, acc);
  }
}

// ---- 4c. segmented accumulation in AFFINE coordinates ("chains") -------------------------------
// Same chunking of the bucket-sorted entry list and same outputs as k_msm_accumulate, but a
// thread walks AFC_J chunks ("chains") in lockstep and keeps their running sums affine.  Step s
// adds entry s of every chain: the AFC_J denominators (x_P - x_acc) are multiplied up, inverted
// ONCE per thread by division steps (fq_inv.cuh: ALU pipe, the multiplier pipe is the bound) and
// unwound with Montgomery's trick, so an addition costs 5M + 1S (+ 1/AFC_J inversion) = ~1.7e3
// wide multiplies against 2.7e3 for the XYZZ mixed addition.  The running sums live in global
// memory (96 B read + written per addition; HBM is ~3 % utilised by this kernel), the prefix
// products in thread-local memory.  No pairing pass, no sorting by size, no intermediate lists.
// kinds: 0 chord, 1 tangent, 2 sum is the identity, 3 nothing to add, 4 first point of a run.
#define AFC_J 16
#ifndef AFC_MIN_BLOCKS
#define AFC_MIN_BLOCKS 4
#endif
// One shared copy of the multiplier / squarer: the three phases of the kernel (collect, invert,
// unwind) run in different warps at the same time, so the instruction footprint matters more than a call.
static __device__ __noinline__ Fq afc_mul(Fq a, Fq b) { return fq_mul(a, b); }
static __device__ __noinline__ Fq afc_sqr(Fq a) { return fq_sqr(a); }

__device__ __forceinline__ void afc_flush(G1Xyzz* dst, const G1Affine* acc, bool empty) {
  G1Xyzz o;
  if (empty) {
    o = xyzz_identity();
  } else {
    o.x = fq_load(&acc->x);
    o.y = fq_load(&acc->y);
    o.zz = fq_one();
    o.zzz = fq_one();
  }
  xyzz_store(dst, o);
}

__global__ void __launch_bounds__(128, AFC_MIN_BLOCKS) k_msm_accumulate_affine(const G1Affine* __restrict__ bases,
                                                                  const uint2* __restrict__ sorted,
                                                                  const unsigned* __restrict__ m_ptr, unsigned nchunks,
                                                                  unsigned chunk, G1Affine* __restrict__ acc_buf,
                                                                  G1Xyzz* __restrict__ buckets,
                                                                  unsigned* __restrict__ part_keys,
                                                                  G1Xyzz* __restrict__ part_pts) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned c0 = t * AFC_J;
  if (c0 >= nchunks) return;
  const unsigned m_total = *m_ptr;
  unsigned cur[AFC_J];
  Fq den[AFC_J];   // denominators on the way in, prefix products after the multiply-up
  unsigned first_mask = 0xffffffffu, empty_mask = 0xffffffffu;
#pragma unroll 1
  for (int j = 0; j < AFC_J; j++) {
    const unsigned c = c0 + j;
    const unsigned start = c * chunk;
    cur[j] = (c < nchunks && start < m_total) ? sorted[start].y : MSM_NONE;
  }
#pragma unroll 1
  for (unsigned s = 0; s < chunk; s++) {
    unsigned long long kinds = 0;
    // ---- collect: close finished runs, fetch operands, form the denominators (no products: the
    //      loads of different chains are independent and overlap) ----
#pragma unroll 4
    for (int j = 0; j < AFC_J; j++) {
      const unsigned c = c0 + j;
      const unsigned e = c * chunk + s;
      unsigned kind = 3;
      Fq d = fq_zero();
      if (c < nchunks && e < m_total) {
        const uint2 ent = sorted[e];
        if (ent.y != cur[j]) {
          const bool empty = (empty_mask >> j) & 1;
          if ((first_mask >> j) & 1) {
            part_keys[2 * c] = cur[j];
            afc_flush(part_pts + 2 * c, acc_buf + c, empty);
            first_mask &= ~(1u << j);
          } else {
            afc_flush(buckets + cur[j], acc_buf + c, empty);
          }
          empty_mask |= 1u << j;
          cur[j] = ent.y;
        }
        const G1Affine* pp = bases + (ent.x & 0x7fffffffu);
        const Fq px = fq_load(&pp->x);
        if (fq_is_zero(px) && fq_is_zero(fq_load(&pp->y))) {
          kind = 3;                                   // the SRS holds the identity here
        } else if ((empty_mask >> j) & 1) {
          kind = 4;
        } else {
          d = fq_sub(px, fq_load(&acc_buf[c].x));
          kind = 0;
          if (fq_is_zero(d)) {                        // same x: doubling or cancellation
            Fq py = fq_load(&pp->y);
            if (ent.x >> 31) py = fq_neg(py);
            const Fq ay = fq_load(&acc_buf[c].y);
            if (fq_eq(py, ay)) {
              d = fq_dbl(ay);
              kind = 1;
            } else {
              kind = 2;
            }
          }
        }
      }
      den[j] = d;
      kinds |= (unsigned long long)kind << (4 * j);
    }
    // ---- multiply up ----
    Fq run = fq_one();
#pragma unroll 1
    for (int j = 0; j < AFC_J; j++) {
      const Fq d = den[j];
      den[j] = run;
      if (((unsigned)(kinds >> (4 * j)) & 15u) <= 1) run = afc_mul(run, d);
    }
    Fq inv = fq_inverse(run);
    // ---- unwind: one affine addition per chain ----
#pragma unroll 1
    for (int j = AFC_J - 1; j >= 0; j--) {
      const unsigned kind = (unsigned)(kinds >> (4 * j)) & 15u;
      if (kind == 3) continue;
      const unsigned c = c0 + j;
      if (kind == 2) {
        empty_mask |= 1u << j;
        continue;
      }
      const uint2 ent = sorted[c * chunk + s];
      G1Affine p = affine_load(bases + (ent.x & 0x7fffffffu));
      if (ent.x >> 31) p.y = fq_neg(p.y);
      G1Affine* ap = acc_buf + c;
      if (kind == 4) {
        fq_store(&ap->x, p.x);
        fq_store(&ap->y, p.y);
        empty_mask &= ~(1u << j);
        continue;
      }
      const G1Affine a = affine_load(ap);
      Fq d, num;
      if (kind == 0) {
        d = fq_sub(p.x, a.x);
        num = fq_sub(p.y, a.y);
      } else {
        d = fq_dbl(a.y);
        const Fq xx = afc_sqr(a.x);
        num = fq_add(fq_dbl(xx), xx);
      }
      const Fq dinv = afc_mul(inv, den[j]);
      inv = afc_mul(inv, d);
      const Fq lam = afc_mul(num, dinv);
      const Fq x3 = fq_sub(fq_sub(afc_sqr(lam), a.x), p.x);
      const Fq y3 = fq_sub(afc_mul(lam, fq_sub(a.x, x3)), a.y);
      fq_store(&ap->x, x3);
      fq_store(&ap->y, y3);
    }
  }
  // ---- head / tail partials of every chain (same contract as k_msm_accumulate) ----
#pragma unroll 1
  for (int j = 0; j < AFC_J; j++) {
    const unsigned c = c0 + j;
    if (c >= nchunks) break;
    if (c * chunk >= m_total) {
      part_keys[2 * c] = MSM_NONE | MSM_IDENT;
      part_keys[2 * c + 1] = MSM_NONE | MSM_IDENT;
      continue;
    }
    const bool empty = (empty_mask >> j) & 1;
    if ((first_mask >> j) & 1) {
      part_keys[2 * c] = cur[j];
      afc_flush(part_pts + 2 * c, acc_buf + c, empty);
      part_keys[2 * c + 1] = cur[j] | MSM_IDENT;
    } else {
      part_keys[2 * c + 1] = cur[j];
      afc_flush(part_pts + 2 * c + 1, acc_buf + c, empty);
    }
  }
}

// ---- 5a. boundary fix-up, common case ---------------------------------------------------------
// A chunk's head run is complete if it starts in that chunk and the chunk has further runs.  The
// run that is still open at the end of chunk t (its tail, or its head when the whole chunk is one
// run that starts there) is owned by thread t, which walks forward over the heads of the following
// chunks until the run ends.  The host takes this path when the largest bucket is shorter than
// PAIR_MAX_SPAN chunks, so the walk is at most PAIR_MAX_SPAN + 1 additions and almost always one;
// heavier skew goes through the logarithmic merge below.
#define PAIR_MAX_SPAN 8
template <bool LAZY>
__global__ void __launch_bounds__(128) k_msm_pair_fixup(const unsigned* __restrict__ part_keys,
                                                        const G1Xyzz* __restrict__ part_pts, unsigned nchunks,
                                                        G1Xyzz* __restrict__ buckets) {
  unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nchunks) return;
  const unsigned hk = part_keys[2 * t];
  if ((hk & MSM_NONE) == MSM_NONE) return;  // chunk beyond the live list
  const unsigned lraw = part_keys[2 * t + 1];
  const bool multi = !(lraw & MSM_IDENT);
  const bool head_starts = t == 0 || (part_keys[2 * t - 1] & MSM_NONE) != hk;
  if (head_starts && multi) {  // complete run: copy
    G1Xyzz h = xyzz_load(part_pts + 2 * t);
    xyzz_store(buckets + hk, h);
  }
  if (!multi && !head_starts) return;  // interior piece of a run owned by an earlier chunk
  const unsigned key = multi ? lraw : hk;
  G1Xyzz acc = xyzz_load(part_pts + 2 * t + (multi ? 1 : 0));
  for (unsigned j = t + 1; j < nchunks && part_keys[2 * j] == key; j++) {
    G1Xyzz h = xyzz_load(part_pts + 2 * j);
    xyzz_add<LAZY>(acc, h);
    if (!(part_keys[2 * j + 1] & MSM_IDENT)) break;  // chunk j has further runs: this one ended there
  }
  xyzz_store(buckets + key, acc);
}

// ---- 5b. boundary merge -----------------------------------------------------------------------
// The partial list (2 slots per chunk, keys non-decreasing) is reduced level by level: every
// thread takes MERGE_B consecutive slots, sums runs of equal key with general XYZZ additions,
// writes runs that lie strictly inside its block to their bucket (it is their only owner) and
// emits a head / tail partial for the next level.  Run length -- i.e. bucket size -- only costs
// extra levels of ~MERGE_B additions, so a bucket holding millions of points (small top window,
// repeated scalars) is as parallel as a uniform one.  The last level is one thread.
#define MERGE_B 16
template <bool LAZY>
__global__ void __launch_bounds__(128) k_msm_merge_level(const unsigned* __restrict__ keys_in,
                                                         const G1Xyzz* __restrict__ pts_in, unsigned nslots,
                                                         G1Xyzz* __restrict__ buckets, unsigned* __restrict__ keys_out,
                                                         G1Xyzz* __restrict__ pts_out, int final_level) {
  unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned start = final_level ? 0 : t * MERGE_B;
  if (start >= nslots || (final_level && t != 0)) return;
  unsigned end = final_level ? nslots : (start + MERGE_B < nslots ? start + MERGE_B : nslots);
  unsigned k0 = keys_in[start];
  unsigned cur = k0 & MSM_NONE;
  G1Xyzz acc = (k0 & MSM_IDENT) ? xyzz_identity() : xyzz_load(pts_in + start);
  bool is_first_run = true;
  for (unsigned e = start + 1; e < end; e++) {
    unsigned kraw = keys_in[e];
    unsigned key = kraw & MSM_NONE;
    if (key != cur) {
      if (is_first_run && !final_level) {
        keys_out[2 * t] = cur;
        xyzz_store(pts_out + 2 * t, acc);
        is_first_run = false;
      } else if (cur != MSM_NONE) {
        xyzz_store(buckets + cur, acc);
      }
      cur = key;
      acc = (kraw & MSM_IDENT) ? xyzz_identity() : xyzz_load(pts_in + e);
    } else if (!(kraw & MSM_IDENT)) {
      G1Xyzz o = xyzz_load(pts_in + e);
      xyzz_add<LAZY>(acc, o);
    }
  }
  if (final_level) {
    if (cur != MSM_NONE) xyzz_store(buckets + cur, acc);
  } else if (is_first_run) {
    keys_out[2 * t] = cur;
    xyzz_store(pts_out + 2 * t, acc);
    keys_out[2 * t + 1] = cur | MSM_IDENT;
  } else {
    keys_out[2 * t + 1] = cur;
    xyzz_store(pts_out + 2 * t + 1, acc);
  }
}

// ---- 6. bucket reduction ---------------------------------------------------------------------
// Wanted per bucket set: V = sum_b (b + 1) * B_b = P + F(B), with P = sum_b B_b and
// F(A) = sum_m m * A_m.  Writing m = S * seg + j:
//     F(A) = sum_seg t_seg + S * F(R),   t_seg = sum_j j * A[S seg + j],  R_seg = sum_j A[S seg + j]
// k_msm_wsum_level computes (t_seg, R_seg) with running sums (2 additions per element, every lane busy) and
// shrinks the array S-fold; the plain sum T = sum_seg t_seg and F(R) are left to the tree-sum kernels below.
// No thread ever does a scalar multiplication.
#define WSUM_S_FIRST 16      // segment length of the first running-sum level (where the work is)
#define WSUM_S_NEXT 8        // and of the later ones
#define WSUM_MAX_LEVELS 4
#ifndef TP_WSUM_MIN_BLOCKS
#define TP_WSUM_MIN_BLOCKS 3   // 168 registers; 4 blocks (128 registers, 36 bytes of spills): reduce +0.27 ms, 5: +0.7 (profiles r2 J)
#endif
template <bool LAZY>
__global__ void __launch_bounds__(128, TP_WSUM_MIN_BLOCKS) k_msm_wsum_level(const G1Xyzz* __restrict__ in, const unsigned* __restrict__ hist,
                                                        unsigned m_in, unsigned seg, unsigned total_out,
                                                        G1Xyzz* __restrict__ r_out, G1Xyzz* __restrict__ t_out) {
  unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total_out) return;
  const unsigned m_out = m_in / seg;
  const size_t base = (size_t)(t / m_out) * m_in + (size_t)(t % m_out) * seg;
  G1Xyzz running = xyzz_identity(), tot = xyzz_identity();
  for (int j = (int)seg - 1; j >= 0; j--) {
    if (!hist || hist[base + j] != 0) {  // first level: empty buckets were never written
      G1Xyzz p = xyzz_load(in + base + j);
      xyzz_add<LAZY>(running, p);
    }
    if (j > 0) xyzz_add<LAZY>(tot, running);
  }
  xyzz_store(r_out + t, running);
  xyzz_store(t_out + t, tot);
}

// Tree sums.  What the running-sum levels leave (or, for a small bucket set, the raw buckets themselves) is an array
// A of m entries per set, viewed as a rows x cols matrix, entry index = cols * hi + lo.  With the row sums
// D[hi] = sum_lo A[hi, lo] and the column sums C[lo] = sum_hi A[hi, lo],
//     F(A) = sum_i i A_i = F(C) + cols * F(D),      P = sum_i A_i = sum_hi D[hi]
// -- two additions per entry again, but as tree sums whose longest dependent chain is cols / 64 + 6 additions instead
// of the 2 S of a running-sum level: that chain is what a small (sharded, or single-MSM) bucket set is bound by.
// The short arrays D and C are then finished bit by bit, F(X) = sum_k 2^k (sum of the X_i with bit k of i set).
// Both stages are lists of JOBS of one shape -- sum `count` entries `stride` apart, optionally only those whose
// index has a given bit set, optionally skipping buckets the histogram says were never written -- one block per
// (job, set); a stage is one launch.
#define TS_THREADS 64
#define TS_MAX_TASKS 32
struct TreeTask {
  const G1Xyzz* src;      // first entry of job 0 of set 0
  const unsigned* hist;   // parallel to src (raw buckets) or null
  G1Xyzz* dst;            // result of job 0 of set 0
  size_t set_stride;      // entries between the sets of src
  unsigned dst_set_stride;
  unsigned njobs;         // jobs per set
  unsigned job_stride;    // entries between the first entries of consecutive jobs
  unsigned count, stride; // entries a job sums and their distance
  int bit;                // >= 0: only entries whose index (0 .. count) has this bit set; for such tasks njobs == 1
};
struct TreeTasks {
  TreeTask t[TS_MAX_TASKS];
  unsigned first[TS_MAX_TASKS + 1];  // block index of each task's job 0
  int ntasks;
};
// LAZY: the sums come out normalised to [0, q) -- what the host (or, sharded, k_msm_combine) reads is canonical.
template <bool LAZY>
__global__ void __launch_bounds__(TS_THREADS) k_msm_treesum(TreeTasks tasks) {
  __shared__ G1Xyzz sh[TS_THREADS];
  int k = 0;
  while (k + 1 < tasks.ntasks && blockIdx.x >= tasks.first[k + 1]) k++;
  const TreeTask& tk = tasks.t[k];
  const unsigned job = blockIdx.x - tasks.first[k], set = blockIdx.y;
  const size_t base = (size_t)set * tk.set_stride + (size_t)job * tk.job_stride;
  const G1Xyzz* src = tk.src + base;
  const unsigned* h = tk.hist ? tk.hist + base : nullptr;
  G1Xyzz acc = xyzz_identity();
  for (unsigned i = threadIdx.x; i < tk.count; i += TS_THREADS) {
    if (tk.bit >= 0 && !((i >> tk.bit) & 1)) continue;
    const size_t e = (size_t)i * tk.stride;
    if (h && h[e] == 0) continue;   // raw buckets: empty ones were never written
    G1Xyzz p = xyzz_load(src + e);
    xyzz_add<LAZY>(acc, p);
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (unsigned d = TS_THREADS / 2; d > 0; d >>= 1) {
    if (threadIdx.x < d) {
      G1Xyzz a = sh[threadIdx.x];
      G1Xyzz b = sh[threadIdx.x + d];
      xyzz_add<LAZY>(a, b);
      sh[threadIdx.x] = a;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) xyzz_store(tk.dst + (size_t)set * tk.dst_set_stride + job, LAZY ? xyzz_norm2(sh[0]) : sh[0]);
}

// ---- 7. cross-rank combination (sharded MSM) --------------------------------------------------------
// `gathered` holds every rank's reduction output: rank r's [sets][slots] block of this job starts at r * rank_stride
// (the all-gather of msm_winsums, which carries all jobs of a batch).  The tail the
// host runs per bucket set is linear in the slots and, except for slot 0 (P = sum of the rank's buckets, which enters
// with the rank-dependent factor rank + 1), the same on every rank: slots >= 1 are therefore summed over ranks here --
// one warp per (set, slot), lane r holding rank r's point, a shared-memory tree -- and the `world` P points pass
// through.  out: [sets][(slots - 1) sums | world P points].  LAZY: the inputs come canonical from k_msm_treesum, the sums
// are normalised back to [0, q) before the host reads them.
template <bool LAZY>
__global__ void __launch_bounds__(32) k_msm_combine(const G1Xyzz* __restrict__ gathered, unsigned world, unsigned rank_stride,
                                                    unsigned slots, G1Xyzz* __restrict__ out) {
  __shared__ G1Xyzz sh[32];
  const unsigned set = blockIdx.x / slots, slot = blockIdx.x % slots;
  const unsigned width = slots - 1 + world;
  const unsigned r = threadIdx.x;
  G1Xyzz p = xyzz_identity();
  if (r < world) p = xyzz_load(gathered + (size_t)r * rank_stride + (size_t)set * slots + slot);
  if (slot == 0) {
    if (r < world) xyzz_store(out + (size_t)set * width + (slots - 1) + r, p);
    return;
  }
  sh[r] = p;
  __syncwarp();
  for (unsigned d = 16; d > 0; d >>= 1) {
    if (r < d && r + d < world) {
      G1Xyzz a = sh[r];
      G1Xyzz b = sh[r + d];
      xyzz_add<LAZY>(a, b);
      sh[r] = a;
    }
    __syncwarp();
  }
  if (r == 0) xyzz_store(out + (size_t)set * width + (slot - 1), LAZY ? xyzz_norm2(sh[0]) : sh[0]);
}

// ---- host side ---------------------------------------------------------------------------------
void encode_g1(const tph::HG1& p, uint8_t out[TP_G1_BYTES]) {
  tph::HFq x, y;
  if (tph::g1_to_affine(p, &x, &y)) {
    memcpy(out, x.v, 48);
    memcpy(out + 48, y.v, 48);
    out[96] = 0;
  } else {
    tph::HFq zero = tph::HFq::zero(), one = tph::HFq::one();
    memcpy(out, zero.v, 48);
    memcpy(out + 48, one.v, 48);
    out[96] = 1;
  }
}

// Affine conversion of a whole batch with ONE field inversion (Montgomery's trick): the inversion is ~570 field
// products on the host, a commitment batch has up to nine of them back to back.  Same bytes as encode_g1.
static void encode_g1_batch(const tph::HG1* p, uint8_t (*out)[TP_G1_BYTES], int n) {
  tph::HFq prefix[MSM_MAX_BATCH];
  tph::HFq run = tph::HFq::one();
  for (int i = 0; i < n; i++) {
    prefix[i] = run;
    if (!p[i].is_identity()) run = run * p[i].z;
  }
  tph::HFq inv = run.inv();
  for (int i = n - 1; i >= 0; i--) {
    if (p[i].is_identity()) {
      encode_g1(p[i], out[i]);
      continue;
    }
    const tph::HFq zi = inv * prefix[i];
    inv = inv * p[i].z;
    const tph::HFq zi2 = zi.sqr();
    const tph::HFq x = p[i].x * zi2, y = p[i].y * zi2 * zi;
    memcpy(out[i], x.v, 48);
    memcpy(out[i] + 48, y.v, 48);
    out[i][96] = 0;
  }
}

template <typename T>
static int exclusive_scan(tp_ctx* ctx, const T* in, T* out, size_t n, unsigned* max_out) {
  size_t nblocks = (n + SCAN_BLOCK - 1) / SCAN_BLOCK;
  TP_TRY(ensure(ctx, ctx->msm_blocksums, nblocks * sizeof(T)));
  T* sums = (T*)ctx->msm_blocksums.p;
  k_scan_local<T><<<(unsigned)nblocks, SCAN_BLOCK, 0, ctx->stream>>>(in, out, sums, n, max_out);
  TP_LAUNCH(ctx, "k_scan_local");
  k_scan_sums<T><<<1, SCAN_BLOCK, 0, ctx->stream>>>(sums, nblocks);
  TP_LAUNCH(ctx, "k_scan_sums");
  k_scan_add<T><<<(unsigned)nblocks, SCAN_BLOCK, 0, ctx->stream>>>(out, sums, n);
  TP_LAUNCH(ctx, "k_scan_add");
  return TP_OK;
}

// ---- pipeline ------------------------------------------------------------------------------------------------------
// An MSM is three kinds of work: a sort bound by atomics and random stores, an accumulation (and the first
// running-sum level of the reduction) bound by the wide-multiply pipe, and latency-bound tails (boundary fix-up, tree
// sums) that keep a few hundred threads busy.  Run back to back on one stream, the first and the last leave the
// multiplier idle: 7 of 82 ms of a 2^20 proof.  A batch is therefore cut into SUB-BATCHES (jobs) that travel through
// three streams -- sort (high priority), accumulate + running sums (normal priority), tails (high priority) -- linked
// by events, each job on its own LANE of scratch buffers:
//
//     sort:   S0 S1       S2
//     acc:       A0 ------A1 ------ W0  A2 ------ W1  W2          (W = running-sum levels of the reduction)
//     tails:              F0        F1  T0        F2  T1  T2      (F = boundary fix-up, T = tree sums)
//
// so the sort and the tails of one job run underneath the accumulation of its neighbours; the high priority makes the
// block scheduler place their (few, small) blocks ahead of the accumulation's pending ones as SM slots come free.  The
// host waits once per job for the sort's two counters (live entries, largest bucket: they size the accumulation) --
// while the previous job accumulates -- and once at the end for ALL jobs' reduction outputs, which share one buffer:
// one all-gather (sharded), one copy to the host, then the serial tails on host threads.
// msm_pipe_submit / msm_pipe_finish expose the two halves so that the prover can queue other work in between
// (api.cu: the quotient's commitments start while the opening polynomials are still being computed).
// Not overlapped (option msm_pipeline = 0, small inputs, the opt-in affine variants): the same stages run in order
// on the context's stream.
#define MSM_LANES 3
struct MsmLane {
  DevBuf hist, offsets, sorted, buckets, part_keys, part_pts, seg;
  cudaEvent_t ev_sorted = nullptr, ev_acc = nullptr, ev_fix = nullptr, ev_wsum = nullptr, ev_done = nullptr;
  bool busy = false;   // ev_done belongs to a job that may still be running
};
struct MsmJob {
  int lane = 0, batch = 0, first_result = 0;
  size_t len = 0;
  const tp_srs* srs = nullptr;
  MsmPlan pl;
  unsigned nsets_total = 0;
  size_t nkeys = 0;
  unsigned m_total = 0, max_bucket = 0, nchunks = 0;
  bool pair_path = true, empty = false, reduce_queued = false;
  bool lazy = true;      // option msm_fq_lazy when the job was queued: every kernel of the job uses the same laws
  // reduction plan
  int nl = 0;
  unsigned m_level[WSUM_MAX_LEVELS + 1], seg_level[WSUM_MAX_LEVELS + 1], tcount[WSUM_MAX_LEVELS + 1], tjobs[WSUM_MAX_LEVELS + 1];
  unsigned bC = 0, bD = 0, cols = 0, rows = 0, total_masks = 0;
  size_t win_off = 0;    // first slot of this job in msm_winsums
  size_t host_off = 0;   // first slot of this job in the buffer the host reads back
};
struct MsmPipe {
  cudaStream_t s_sort = nullptr, s_acc = nullptr, s_tail = nullptr;
  cudaEvent_t ev_in = nullptr;
  MsmLane lane[MSM_LANES];
  unsigned* counts = nullptr;   // pinned, [lane][2]: live entries, largest bucket
  std::vector<MsmJob> jobs;
  bool overlap = false;         // mode of the batch being queued
  size_t win_used = 0;          // slots of msm_winsums the queued jobs take
  int results = 0;              // results the queued jobs will return
  int next_lane = 0;
  ProfScope* total = nullptr;   // TP_PHASE_MSM_TOTAL of an overlapped batch: first submit to the end of finish
};

// grow-only like ensure(), but the old buffer may be in use on any of the pipe's streams
static int ensure_idle(tp_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return TP_OK;
  if (b.p) TP_CUDA_OK(ctx, cudaDeviceSynchronize());
  return ensure(ctx, b, bytes);
}

static int pipe_get(tp_ctx* ctx, MsmPipe** out) {
  if (!ctx->msm_pipe) {
    MsmPipe* p = new MsmPipe();
    ctx->msm_pipe = p;
    if (cudaMallocHost(&p->counts, MSM_LANES * 2 * sizeof(unsigned)) != cudaSuccess) return fail(ctx, TP_ERR_CUDA, "msm: pinned allocation failed");
    TP_CUDA_OK(ctx, cudaEventCreateWithFlags(&p->ev_in, cudaEventDisableTiming));
    for (auto& l : p->lane)
      for (cudaEvent_t* e : {&l.ev_sorted, &l.ev_acc, &l.ev_fix, &l.ev_wsum, &l.ev_done})
        TP_CUDA_OK(ctx, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  *out = ctx->msm_pipe;
  return TP_OK;
}
static int pipe_streams(tp_ctx* ctx, MsmPipe* p) {
  if (p->s_acc) return TP_OK;
  int least = 0, greatest = 0;
  TP_CUDA_OK(ctx, cudaDeviceGetStreamPriorityRange(&least, &greatest));
  TP_CUDA_OK(ctx, cudaStreamCreateWithPriority(&p->s_sort, cudaStreamNonBlocking, greatest));
  TP_CUDA_OK(ctx, cudaStreamCreateWithPriority(&p->s_tail, cudaStreamNonBlocking, greatest));
  TP_CUDA_OK(ctx, cudaStreamCreateWithPriority(&p->s_acc, cudaStreamNonBlocking, least));
  return TP_OK;
}
void msm_pipe_destroy(tp_ctx* ctx) {
  MsmPipe* p = ctx->msm_pipe;
  if (!p) return;
  cudaDeviceSynchronize();
  for (cudaStream_t s : {p->s_sort, p->s_acc, p->s_tail})
    if (s) cudaStreamDestroy(s);
  if (p->ev_in) cudaEventDestroy(p->ev_in);
  for (auto& l : p->lane) {
    for (DevBuf* b : {&l.hist, &l.offsets, &l.sorted, &l.buckets, &l.part_keys, &l.part_pts, &l.seg}) release(*b);
    for (cudaEvent_t e : {l.ev_sorted, l.ev_acc, l.ev_fix, l.ev_wsum, l.ev_done})
      if (e) cudaEventDestroy(e);
  }
  if (p->counts) cudaFreeHost(p->counts);
  delete p->total;
  delete p;
  ctx->msm_pipe = nullptr;
}
// after an error: nothing of the queued batch survives
static void pipe_abort(tp_ctx* ctx) {
  MsmPipe* p = ctx->msm_pipe;
  if (!p) return;
  cudaDeviceSynchronize();
  p->jobs.clear();
  p->win_used = 0;
  p->results = 0;
  for (auto& l : p->lane) l.busy = false;
  delete p->total;
  p->total = nullptr;
}

static cudaStream_t pipe_sort_stream(tp_ctx* ctx, MsmPipe* p) { return p->overlap ? p->s_sort : ctx->stream; }
static cudaStream_t pipe_acc_stream(tp_ctx* ctx, MsmPipe* p) { return p->overlap ? p->s_acc : ctx->stream; }
static cudaStream_t pipe_tail_stream(tp_ctx* ctx, MsmPipe* p) { return p->overlap ? p->s_tail : ctx->stream; }
static int pipe_wait(tp_ctx* ctx, MsmPipe* p, cudaStream_t s, cudaEvent_t e) {   // one stream when not overlapped: already ordered
  if (p->overlap) TP_CUDA_OK(ctx, cudaStreamWaitEvent(s, e, 0));
  return TP_OK;
}
static int pipe_record(tp_ctx* ctx, MsmPipe* p, cudaEvent_t e, cudaStream_t s) {
  if (p->overlap) TP_CUDA_OK(ctx, cudaEventRecord(e, s));
  return TP_OK;
}

// Inputs worth overlapping: from about 2^15 points the accumulation of a job is long enough to cover its neighbours' sort.
bool msm_pipe_overlaps(const tp_ctx* ctx, size_t len) {
  static const unsigned env_min_log = env_uint("TP_MSM_PIPE_MIN_LOG", 0);
  const unsigned min_log = env_min_log ? env_min_log : ctx->msm_pipe_min_log;
  static const bool env_off = getenv("TP_MSM_PIPELINE") && *getenv("TP_MSM_PIPELINE") == '0';
  static const bool env_all = getenv("TP_MSM_PIPELINE") && *getenv("TP_MSM_PIPELINE") == '2';
  // Off unless asked for.  The accumulation fills every SM's register file (3 x 128 threads x 168 registers) and the
  // planner sizes a sharded rank's chunks so that its smaller grid still covers the whole GPU: a second kernel only
  // gets slots as accumulation blocks retire, so the "overlapped" sort runs no sooner than it would alone, while the
  // smaller sub-batches reduce less efficiently.  2^20 gates: 84.2 ms against 82.2 on one B200, 18.1 against 16.7 on
  // eight; 2^22 on eight: 54.2 against 52.4 (profiles/r2_summary.md I).
  const bool want = ctx->msm_pipeline == 2 || env_all || (ctx->msm_pipeline == 1 && ctx->world > 1);
  return want && !env_off && ctx->msm_aff_rounds == 0 && ctx->msm_affine_chains == 0 && len >= ((size_t)1 << min_log);
}

// ---- stage 1: digits, bucket offsets, counting-sort scatter (sort stream); ends with the two counters on their way to the host
static int job_sort(tp_ctx* ctx, MsmPipe* p, MsmJob& j, const Fr* const* scalars) {
  MsmLane& ln = p->lane[j.lane];
  const MsmPlan& pl = j.pl;
  const unsigned world = ctx->world > 1 ? (unsigned)ctx->world : 1u;
  const size_t len = j.len, nkeys = j.nkeys;
  const size_t total = (size_t)pl.nwin * j.batch * len;
  TP_TRY(ensure_idle(ctx, ln.hist, (nkeys + 2) * sizeof(unsigned)));  // + scan sentinel + largest bucket
  TP_TRY(ensure_idle(ctx, ln.offsets, (nkeys + 1) * sizeof(unsigned)));
  TP_TRY(ensure_idle(ctx, ln.sorted, total * sizeof(uint2)));
  TP_TRY(ensure_idle(ctx, ln.buckets, nkeys * sizeof(G1Xyzz)));
  unsigned* hist = (unsigned*)ln.hist.p;
  unsigned* offsets = (unsigned*)ln.offsets.p;
  uint2* sorted = (uint2*)ln.sorted.p;
  const bool compact = world > 1 && !env_uint("TP_MSM_NO_COMPACT", 0);
  if (compact) TP_TRY(ensure_idle(ctx, ctx->msm_compact, total * sizeof(MsmEntry) + 16));
  if (!compact || ctx->msm_aff_rounds) {   // keys / ranks live from the digit pass to the scatter only: one copy, all sorts run
                                           // on one stream (the opt-in affine rounds reuse the key array as a counter array)
    TP_TRY(ensure_idle(ctx, ctx->msm_keys, total * sizeof(unsigned)));
    TP_TRY(ensure_idle(ctx, ctx->msm_ranks, total * sizeof(unsigned)));
  }
  {
    const size_t nblocks = (nkeys + 1 + SCAN_BLOCK - 1) / SCAN_BLOCK;
    TP_TRY(ensure_idle(ctx, ctx->msm_blocksums, nblocks * sizeof(unsigned)));
  }
  unsigned* keys = (unsigned*)ctx->msm_keys.p;
  unsigned* ranks = (unsigned*)ctx->msm_ranks.p;
  StreamSwap sw(ctx, pipe_sort_stream(ctx, p));
  {
    ProfScope prof(ctx, TP_PHASE_MSM_SORT);
    TP_CUDA_OK(ctx, cudaMemsetAsync(hist, 0, (nkeys + 2) * sizeof(unsigned), ctx->stream));
    MsmScalarSets sets;
    for (int b = 0; b < MSM_MAX_BATCH; b++) sets.p[b] = scalars[b < j.batch ? b : 0];
    dim3 grid((unsigned)((len + 255) / 256), (unsigned)j.batch);
    if (compact) {
      // sharded: owned entries into a compact list, scatter over that list (see 1b)
      unsigned* list_count = (unsigned*)ctx->msm_compact.p;
      MsmEntry* list = (MsmEntry*)((char*)ctx->msm_compact.p + 16);
      TP_CUDA_OK(ctx, cudaMemsetAsync(list_count, 0, sizeof(unsigned), ctx->stream));
      MsmOwner own;
      own.world = world;
      own.rank = (unsigned)ctx->rank;
      own.mask = world - 1;
      own.shift = 32;
      if ((world & (world - 1)) == 0) own.shift = (unsigned)__builtin_ctz(world);
      k_msm_digits_sharded<<<grid, 256, 0, ctx->stream>>>(sets, len, pl.c, pl.nwin, pl.nbuck, pl.levels, pl.nsets, own,
                                                          (unsigned)j.srs->len, hist, list_count, list);
      TP_LAUNCH(ctx, "k_msm_digits_sharded");
      TP_TRY(exclusive_scan<unsigned>(ctx, hist, offsets, nkeys + 1, hist + nkeys + 1));
      k_msm_scatter_compact<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(list, list_count, offsets, sorted);
      TP_LAUNCH(ctx, "k_msm_scatter_compact");
    } else {
      k_msm_digits<<<grid, 256, 0, ctx->stream>>>(sets, len, pl.c, pl.nwin, pl.nbuck, pl.levels, pl.nsets, world,
                                                  (unsigned)ctx->rank, hist, keys, ranks);
      TP_LAUNCH(ctx, "k_msm_digits");
      TP_TRY(exclusive_scan<unsigned>(ctx, hist, offsets, nkeys + 1, hist + nkeys + 1));
      // Two slices when that brings one MSM's share of the sorted list (len * nwin entries of 8 bytes) from "about
      // the L2" to "well inside it" (TP_MSM_SCATTER_WINDOW_MB, default 64); every further slice costs a full pass
      // over the keys (~0.5 ms per proof at 2^20) and measured slower (4: +0.3 ms, 8: +2.3 ms), and a list that
      // is several L2s long gains little (2^24: 9.9 -> 9.4 ms with four).  TP_MSM_SCATTER_SLICES forces a count.
      static const unsigned env_slices = env_uint("TP_MSM_SCATTER_SLICES", 0);
      static const unsigned window_mb = env_uint("TP_MSM_SCATTER_WINDOW_MB", 64);
      unsigned log_slices = 0;
      if (env_slices) {
        while ((2u << log_slices) <= env_slices) log_slices++;
      } else {
        const size_t per_msm = (size_t)pl.nwin * len * sizeof(uint2), window = (size_t)window_mb << 20;
        if (per_msm > 2 * window) log_slices = 2;   // several L2s long: four slices still save a little (2^22: 2.51 -> 2.15 ms)
        else if (per_msm > window) log_slices = 1;
      }
      unsigned log_nbuck = 0;
      while ((1u << log_nbuck) < pl.nbuck) log_nbuck++;
      if (world > 1) {   // a rank scatters 1 / world of the list: fewer slices bring it inside the L2
        unsigned lw = 0;
        while ((2u << lw) <= world) lw++;
        log_slices = log_slices > lw ? log_slices - lw : 0;
      }
      if (log_slices > log_nbuck) log_slices = log_nbuck;
      const unsigned slice_shift = log_nbuck - log_slices;
      const size_t per_block = (size_t)256 * 4 * SCATTER_UNROLL;
      for (unsigned sl = 0; sl < (1u << log_slices); sl++) {
        k_msm_scatter<<<(unsigned)((total + per_block - 1) / per_block), 256, 0, ctx->stream>>>(
            keys, ranks, offsets, len, total, pl.nwin, pl.levels, (unsigned)j.srs->len, sorted, pl.nbuck - 1, slice_shift, sl);
        TP_LAUNCH(ctx, "k_msm_scatter");
      }
    }
    unsigned* cnt = p->counts + 2 * j.lane;
    TP_CUDA_OK(ctx, cudaMemcpyAsync(cnt, offsets + nkeys, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA_OK(ctx, cudaMemcpyAsync(cnt + 1, hist + nkeys + 1, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  }
  TP_TRY(pipe_record(ctx, p, ln.ev_sorted, ctx->stream));
  return TP_OK;
}

// ---- stage 2: accumulation (accumulate stream) and boundary fix-up (tail stream), sized from the sort's counters
static int job_accumulate(tp_ctx* ctx, MsmPipe* p, MsmJob& j) {
  MsmLane& ln = p->lane[j.lane];
  const MsmPlan& pl = j.pl;
  const tp_srs* srs = j.srs;
  const size_t nkeys = j.nkeys;
  const G1Affine* bases = srs->g1;              // level k of point i lives at bases[k * srs->len + i]
  unsigned* hist = (unsigned*)ln.hist.p;
  unsigned* offsets = (unsigned*)ln.offsets.p;
  unsigned* keys = (unsigned*)ctx->msm_keys.p;
  uint2* sorted = (uint2*)ln.sorted.p;
  G1Xyzz* buckets = (G1Xyzz*)ln.buckets.p;
  const unsigned m_total = j.m_total;
  StreamSwap sw(ctx, pipe_acc_stream(ctx, p));
  TP_TRY(pipe_wait(ctx, p, ctx->stream, ln.ev_sorted));
  // ---- batch-affine rounds (4a): plan on the host from upper bounds, sizes stay on the device ----
  // bound[r] >= entries before round r + 1: every round leaves ceil(cnt / 2) per bucket.
  // Off by default: on sm_100a the rounds do not beat the XYZZ accumulation they replace (profiles/r1_summary.md K);
  // tp_ctx_set_option("msm_affine_rounds", r) or TP_MSM_AFF_ROUNDS=r turn them on (never overlapped: ctx scratch).
  const unsigned aff_rounds_env = p->overlap ? 0u : ctx->msm_aff_rounds;
  const unsigned aff_disable = aff_rounds_env == 0;
  size_t bound[AFF_MAX_ROUNDS + 1];
  bound[0] = m_total;
  int rounds = 0;
  unsigned max_b = j.max_bucket;
  const size_t split = (size_t)pl.levels * srs->len;  // table indices are < split
  if (!aff_disable) {
    const int want = (int)(aff_rounds_env < AFF_MAX_ROUNDS ? aff_rounds_env : AFF_MAX_ROUNDS);
    while (rounds < want) {
      // a round needs buckets that hold >= 2 entries on average (the key arrays are reused as counters)
      if (bound[rounds] < 2 * nkeys || bound[rounds] < 64) break;
      bound[rounds + 1] = bound[rounds] / 2 + nkeys;
      rounds++;
    }
  }
  size_t scratch_pts = 0;
  for (int r = 1; r <= rounds; r++) scratch_pts += bound[r];
  if (rounds > 0) {
    // memory: the sums of all rounds stay addressable (later rounds and the accumulation read them)
    const size_t need = scratch_pts * sizeof(G1Affine) + bound[1] * sizeof(uint2);
    if (split + scratch_pts >= ((size_t)1 << 31)) {
      rounds = 0;
    } else if (need > ctx->msm_aff_pts.cap + ctx->msm_sorted2.cap) {
      size_t free_b = 0, total_b = 0;
      cudaMemGetInfo(&free_b, &total_b);
      if (need > (free_b + ctx->msm_aff_pts.cap + ctx->msm_sorted2.cap) / 10 * 8) rounds = 0;  // falls back to XYZZ only
    }
  }
  const uint2* final_list = sorted;
  const unsigned* final_m = offsets + nkeys;
  const G1Affine* scratch = nullptr;
  if (rounds > 0) {
    ProfScope prof(ctx, TP_PHASE_MSM_ACCUM);
    TP_TRY(ensure(ctx, ctx->msm_aff_pts, scratch_pts * sizeof(G1Affine)));
    TP_TRY(ensure(ctx, ctx->msm_sorted2, bound[1] * sizeof(uint2)));
    TP_TRY(ensure(ctx, ctx->msm_aff_cnt, nkeys * sizeof(unsigned)));
    TP_TRY(ensure(ctx, ctx->msm_aff_plan, 2 * (nkeys + 1) * sizeof(unsigned long long)));
    G1Affine* sc = (G1Affine*)ctx->msm_aff_pts.p;
    scratch = sc;
    uint2* lists[2] = {sorted, (uint2*)ctx->msm_sorted2.p};
    unsigned* cnts[2] = {hist, (unsigned*)ctx->msm_aff_cnt.p};   // round 1 reads the histogram; it must survive (the
                                                                 // reduction uses it to skip empty buckets), so the
                                                                 // ping-pong writes go to aff_cnt / keys scratch
    unsigned* cnt_alt = keys;  // the digit keys are dead after the scatter: reuse as the second counter array
    unsigned long long* plans[2] = {(unsigned long long*)ctx->msm_aff_plan.p,
                                    (unsigned long long*)ctx->msm_aff_plan.p + (nkeys + 1)};
    const unsigned* off_in = offsets;
    unsigned off_stride = 1;
    const unsigned* cnt_in = hist;
    const unsigned* m_in = offsets + nkeys;
    TP_TRY(ensure(ctx, ctx->msm_aff_rec, (bound[0] / 2 + 1) * sizeof(uint4)));
    uint4* rec = (uint4*)ctx->msm_aff_rec.p;
    size_t region = 0;
    static bool smem_attr[64] = {false};   // a function attribute belongs to a device: a group context has one rank per device
    if (!smem_attr[ctx->device & 63]) {
      TP_CUDA_OK(ctx, cudaFuncSetAttribute(k_aff_round, cudaFuncAttributeMaxDynamicSharedMemorySize, AFF_SMEM));
      smem_attr[ctx->device & 63] = true;
    }
    for (int r = 0; r < rounds; r++) {
      unsigned* cnt_out = (r & 1) ? cnt_alt : cnts[1];
      unsigned long long* plan = plans[r & 1];
      const uint2* l_in = lists[r & 1];
      uint2* l_out = lists[(r + 1) & 1];
      k_aff_plan<<<(unsigned)((nkeys + 1 + 255) / 256), 256, 0, ctx->stream>>>(cnt_in, nkeys, cnt_out, plan);
      TP_LAUNCH(ctx, "k_aff_plan");
      TP_TRY(exclusive_scan<unsigned long long>(ctx, plan, plan, nkeys + 1, nullptr));
      const size_t pair_bound = bound[r] / 2;
      k_aff_records<<<(unsigned)((bound[r] + 255) / 256), 256, 0, ctx->stream>>>(l_in, m_in, cnt_in, off_in, off_stride, plan,
                                                                                 rec, l_out);
      TP_LAUNCH(ctx, "k_aff_records");
      // pairs per thread: as many as the local arrays hold, fewer when that fills whole waves of the GPU more evenly
      const size_t wave = (size_t)ctx->sm_count * 4 * AFF_THREADS;  // resident threads
      size_t waves = (pair_bound + wave * AFF_K - 1) / (wave * AFF_K);
      unsigned k_run = (unsigned)((pair_bound + waves * wave - 1) / (waves * wave));
      static unsigned k_env = env_uint("TP_MSM_AFF_K", 0);
      if (k_env) k_run = k_env;
      if (k_run > AFF_K) k_run = AFF_K;
      if (k_run < 8) k_run = 8;
      const unsigned nblocks = (unsigned)((pair_bound + (size_t)k_run * AFF_THREADS - 1) / ((size_t)k_run * AFF_THREADS));
      k_aff_round<<<nblocks ? nblocks : 1, AFF_THREADS, AFF_SMEM, ctx->stream>>>(bases, sc, (unsigned)split, rec, plan,
                                                                                 (unsigned)nkeys, l_out, (unsigned)region, k_run);
      TP_LAUNCH(ctx, "k_aff_round");
      m_in = (const unsigned*)(plan + nkeys) + 1;
      region += bound[r + 1];
      cnt_in = cnt_out;
      off_in = (const unsigned*)plan + 1;   // high halves of the scanned plan = offsets of the next list
      off_stride = 2;
      final_list = l_out;
      final_m = (const unsigned*)(plan + nkeys) + 1;
      max_b = (max_b + 1) / 2;
    }
  }
  // Entries per accumulate thread: longer chunks when buckets are long (fewer boundary partials),
  // as long as the grid still fills the GPU several times over.
  const size_t m_bound = bound[rounds];
  unsigned chunk = rounds > 0 ? 16 : msm_chunk();
  while (chunk <= max_b && chunk < 1024 && m_bound / (2 * chunk) >= (size_t)ctx->sm_count * 384 * 4) chunk *= 2;
  // Whole waves: with 3 x 128 resident threads per SM a grid of 1.1 waves costs two; when only a few waves are
  // in play, resize the chunks so that the thread count is a multiple of what the GPU holds at once.
  if (rounds == 0 && !env_uint("TP_MSM_CHUNK", 0)) {
    const double resident = (double)ctx->sm_count * 128 * TP_ACC_MIN_BLOCKS;
    const double waves = (double)m_bound / (resident * chunk);
    if (waves < 8.0) {
      const double w = waves < 1.0 ? 1.0 : (double)(unsigned)(waves + 0.5);
      size_t ch = (size_t)((double)m_bound / (w * resident)) + 1;
      chunk = ch < 32 ? 32u : (ch > 1024 ? 1024u : (unsigned)ch);
    }
  }
  // affine chains (4c): AFC_J chunks per thread, so the chunks shrink until the grid fills the GPU
  const bool chains = rounds == 0 && !p->overlap && ctx->msm_affine_chains != 0;
  if (chains) {
    static unsigned chunk_env = env_uint("TP_MSM_AFC_CHUNK", 0);
    const size_t want = (size_t)ctx->sm_count * 128 * AFC_MIN_BLOCKS * AFC_J;
    size_t ch = m_bound / want;
    chunk = ch < 16 ? 16u : (ch > 64 ? 64u : (unsigned)ch);
    if (chunk_env) chunk = chunk_env;
  }
  j.pair_path = max_b < PAIR_MAX_SPAN * chunk && !msm_force_levels();
  const unsigned nchunks = (unsigned)((m_bound + chunk - 1) / chunk);
  j.nchunks = nchunks;
  // first half: accumulate's partials; second half: ping-pong space for the merge levels
  TP_TRY(ensure_idle(ctx, ln.part_keys, ((size_t)2 * nchunks + (size_t)nchunks / 4 + 64) * sizeof(unsigned)));
  TP_TRY(ensure_idle(ctx, ln.part_pts, ((size_t)2 * nchunks + (size_t)nchunks / 4 + 64) * sizeof(G1Xyzz)));
  ctx->stat_msm_entries += (double)m_total;
  ctx->stat_msm_calls += j.batch;
  ctx->stat_msm_c = pl.c;
  ctx->stat_msm_nwin = pl.nwin;
  ctx->stat_msm_levels = pl.levels;
  ctx->stat_msm_chunk = chunk;
  if (m_total > 0) {
    {
      ProfScope prof(ctx, TP_PHASE_MSM_ACCUM);
      if (chains) {
        TP_TRY(ensure(ctx, ctx->msm_aff_pts, (size_t)nchunks * sizeof(G1Affine)));
        const unsigned nthreads = (nchunks + AFC_J - 1) / AFC_J;
        k_msm_accumulate_affine<<<(nthreads + 127) / 128, 128, 0, ctx->stream>>>(
            bases, final_list, final_m, nchunks, chunk, (G1Affine*)ctx->msm_aff_pts.p, buckets, (unsigned*)ln.part_keys.p,
            (G1Xyzz*)ln.part_pts.p);
        TP_LAUNCH(ctx, "k_msm_accumulate_affine");
      } else {
        const auto acc_kernel = ctx->msm_acc_staged ? (j.lazy ? k_msm_accumulate<true, true> : k_msm_accumulate<true, false>)
                                                    : (j.lazy ? k_msm_accumulate<false, true> : k_msm_accumulate<false, false>);
        acc_kernel<<<(nchunks + ACC_THREADS - 1) / ACC_THREADS, ACC_THREADS, 0, ctx->stream>>>(
            bases, scratch, (unsigned)split, final_list, final_m, nchunks, buckets, (unsigned*)ln.part_keys.p,
            (G1Xyzz*)ln.part_pts.p, chunk);
        TP_LAUNCH(ctx, "k_msm_accumulate");
      }
    }
    TP_TRY(pipe_record(ctx, p, ln.ev_acc, ctx->stream));
    // boundary partials -> buckets, on the tail stream
    StreamSwap st(ctx, pipe_tail_stream(ctx, p));
    TP_TRY(pipe_wait(ctx, p, ctx->stream, ln.ev_acc));
    {
      ProfScope prof(ctx, TP_PHASE_MSM_REDUCE);
      if (j.pair_path) {
        (j.lazy ? k_msm_pair_fixup<true> : k_msm_pair_fixup<false>)<<<(nchunks + 63) / 64, 64, 0, ctx->stream>>>((const unsigned*)ln.part_keys.p, (const G1Xyzz*)ln.part_pts.p,
                                                                      nchunks, buckets);
        TP_LAUNCH(ctx, "k_msm_pair_fixup");
      } else {
        unsigned* ka = (unsigned*)ln.part_keys.p;
        G1Xyzz* pa = (G1Xyzz*)ln.part_pts.p;
        unsigned* kb = ka + 2 * (size_t)nchunks;
        G1Xyzz* pb = pa + 2 * (size_t)nchunks;
        unsigned nslots = 2 * nchunks;
        const auto merge = j.lazy ? k_msm_merge_level<true> : k_msm_merge_level<false>;
        while (nslots > 2 * MERGE_B) {
          unsigned nth = (nslots + MERGE_B - 1) / MERGE_B;
          merge<<<(nth + 127) / 128, 128, 0, ctx->stream>>>(ka, pa, nslots, buckets, kb, pb, 0);
          TP_LAUNCH(ctx, "k_msm_merge_level");
          std::swap(ka, kb);
          std::swap(pa, pb);
          nslots = 2 * nth;
        }
        merge<<<1, 32, 0, ctx->stream>>>(ka, pa, nslots, buckets, kb, pb, 1);
        TP_LAUNCH(ctx, "k_msm_merge_level");
      }
    }
    TP_TRY(pipe_record(ctx, p, ln.ev_fix, ctx->stream));
  } else {
    // a sharded rank that owns none of the digits: its buckets are all empty (the histogram says so)
    TP_TRY(pipe_record(ctx, p, ln.ev_fix, ctx->stream));
  }
  return TP_OK;
}

// Reduction plan.  Running-sum levels (every lane busy, two additions per entry, but a chain of 2 S dependent
// additions per thread) while the batch still has entries enough to keep the whole GPU busy with them -- 16-bucket
// segments first, 8 after that -- then the tree sums.  A small bucket set (a sharded rank's share, a single small
// MSM) is latency-bound from the start and goes straight to the tree sums.
static void job_plan_reduce(const tp_ctx* ctx, MsmJob& j) {
  static const unsigned env_l1 = env_uint("TP_MSM_REDUCE_L1", 0);   // 1: no running-sum level, 2: as many as fit
  const unsigned l1_mode = ctx->msm_reduce_l1 ? ctx->msm_reduce_l1 : env_l1;
  int nl = 0;
  j.m_level[0] = j.pl.nbuck;
  j.seg_level[0] = 1;
  while (nl < WSUM_MAX_LEVELS) {
    const unsigned sg = nl == 0 ? WSUM_S_FIRST : WSUM_S_NEXT;
    if (j.m_level[nl] < 2 * sg || l1_mode == 1) break;
    if (l1_mode != 2 && (size_t)j.nsets_total * j.m_level[nl] < ((size_t)1 << (nl == 0 ? 19 : 18))) break;
    j.seg_level[nl + 1] = sg;
    j.m_level[nl + 1] = j.m_level[nl] / sg;
    nl++;
  }
  j.nl = nl;
  const unsigned m_rc = j.m_level[nl];   // length of the array the row / column sums run over
  unsigned log_m = 0;
  while ((1u << log_m) < m_rc) log_m++;
  j.bC = (log_m + 1) / 2;
  j.bD = log_m - j.bC;
  j.cols = 1u << j.bC;
  j.rows = 1u << j.bD;
  j.total_masks = 1 + j.bD + j.bC + (unsigned)nl;   // [P, bits of D, bits of C, T_1 .. T_nl]
  // the t array of level l (m_level[l] entries per set) only needs its plain sum: first per run of tcount[l] entries
  for (int l = 1; l <= nl; l++) {
    j.tcount[l] = j.m_level[l] > 256 ? 256u : j.m_level[l];
    j.tjobs[l] = j.m_level[l] / j.tcount[l];
  }
}

// ---- stage 3: bucket reduction -- running-sum levels on the accumulate stream, tree sums on the tail stream -------
static int job_reduce(tp_ctx* ctx, MsmPipe* p, MsmJob& j) {
  j.reduce_queued = true;
  if (j.empty) return TP_OK;
  MsmLane& ln = p->lane[j.lane];
  const unsigned nsets_total = j.nsets_total;
  const int nl = j.nl;
  const unsigned rows = j.rows, cols = j.cols, bD = j.bD, bC = j.bC, total_masks = j.total_masks;
  const unsigned m_rc = j.m_level[nl];
  size_t slab = (size_t)nsets_total * (rows + cols);
  for (int l = 1; l <= nl; l++) slab += 2 * (size_t)nsets_total * j.m_level[l] + (size_t)nsets_total * j.tjobs[l];
  TP_TRY(ensure_idle(ctx, ln.seg, slab * sizeof(G1Xyzz)));
  G1Xyzz* cursor = (G1Xyzz*)ln.seg.p;
  const G1Xyzz* cur_in = (const G1Xyzz*)ln.buckets.p;
  const unsigned* cur_hist = (const unsigned*)ln.hist.p;
  const G1Xyzz* t_arr[WSUM_MAX_LEVELS + 1] = {nullptr};
  {
    StreamSwap sw(ctx, pipe_acc_stream(ctx, p));
    TP_TRY(pipe_wait(ctx, p, ctx->stream, ln.ev_fix));
    {
      ProfScope prof(ctx, TP_PHASE_MSM_REDUCE);
      for (int l = 1; l <= nl; l++) {
        const unsigned total_out = nsets_total * j.m_level[l];
        G1Xyzz* r_out = cursor;
        G1Xyzz* t_out = cursor + total_out;
        cursor += 2 * (size_t)total_out;
        (j.lazy ? k_msm_wsum_level<true> : k_msm_wsum_level<false>)<<<(total_out + 127) / 128, 128, 0, ctx->stream>>>(cur_in, cur_hist, j.m_level[l - 1], j.seg_level[l],
                                                                           total_out, r_out, t_out);
        TP_LAUNCH(ctx, "k_msm_wsum_level");
        cur_in = r_out;
        cur_hist = nullptr;
        t_arr[l] = t_out;
      }
    }
    if (nl > 0) TP_TRY(pipe_record(ctx, p, ln.ev_wsum, ctx->stream));
  }
  StreamSwap sw(ctx, pipe_tail_stream(ctx, p));
  TP_TRY(pipe_wait(ctx, p, ctx->stream, nl > 0 ? ln.ev_wsum : ln.ev_fix));
  {
    ProfScope prof(ctx, TP_PHASE_MSM_REDUCE);
    G1Xyzz* D = cursor;
    G1Xyzz* C = D + (size_t)nsets_total * rows;
    cursor = C + (size_t)nsets_total * cols;
    G1Xyzz* TPs[WSUM_MAX_LEVELS + 1] = {nullptr};
    for (int l = 1; l <= nl; l++) {
      TPs[l] = cursor;
      cursor += (size_t)nsets_total * j.tjobs[l];
    }
    auto add_task = [](TreeTasks& tt, const G1Xyzz* src, const unsigned* h, G1Xyzz* dst, size_t set_stride, unsigned dst_set_stride,
                       unsigned njobs, unsigned job_stride, unsigned count, unsigned stride, int bit) {
      TreeTask& k = tt.t[tt.ntasks];
      k.src = src; k.hist = h; k.dst = dst; k.set_stride = set_stride; k.dst_set_stride = dst_set_stride;
      k.njobs = njobs; k.job_stride = job_stride; k.count = count; k.stride = stride; k.bit = bit;
      tt.first[tt.ntasks + 1] = tt.first[tt.ntasks] + njobs;
      tt.ntasks++;
    };
    // stage A: row sums, column sums, partial sums of every level's t array
    TreeTasks ta;
    memset(&ta, 0, sizeof(ta));
    add_task(ta, cur_in, cur_hist, D, m_rc, rows, rows, cols, cols, 1, -1);
    add_task(ta, cur_in, cur_hist, C, m_rc, cols, cols, 1, rows, cols, -1);
    for (int l = 1; l <= nl; l++) add_task(ta, t_arr[l], nullptr, TPs[l], j.m_level[l], j.tjobs[l], j.tjobs[l], j.tcount[l], j.tcount[l], 1, -1);
    const auto treesum = j.lazy ? k_msm_treesum<true> : k_msm_treesum<false>;
    treesum<<<dim3(ta.first[ta.ntasks], nsets_total), TS_THREADS, 0, ctx->stream>>>(ta);
    TP_LAUNCH(ctx, "k_msm_treesum");
    // stage B: one slot each -- P, the bit sums of D and of C, the totals of the t arrays
    G1Xyzz* fin = (G1Xyzz*)ctx->msm_winsums.p + j.win_off;
    struct Slot { const G1Xyzz* src; size_t set_stride; unsigned count; int bit; };
    std::vector<Slot> slots;
    slots.push_back({D, rows, rows, -1});
    for (unsigned k = 0; k < bD; k++) slots.push_back({D, rows, rows, (int)k});
    for (unsigned k = 0; k < bC; k++) slots.push_back({C, cols, cols, (int)k});
    for (int l = 1; l <= nl; l++) slots.push_back({TPs[l], j.tjobs[l], j.tjobs[l], -1});
    for (size_t s0 = 0; s0 < slots.size(); s0 += TS_MAX_TASKS) {
      TreeTasks tb;
      memset(&tb, 0, sizeof(tb));
      for (size_t q = s0; q < slots.size() && q < s0 + TS_MAX_TASKS; q++)
        add_task(tb, slots[q].src, nullptr, fin + q, slots[q].set_stride, total_masks, 1, 0, slots[q].count, 1, slots[q].bit);
      treesum<<<dim3(tb.first[tb.ntasks], nsets_total), TS_THREADS, 0, ctx->stream>>>(tb);
      TP_LAUNCH(ctx, "k_msm_treesum");
    }
  }
  TP_TRY(pipe_record(ctx, p, ln.ev_done, ctx->stream));
  return TP_OK;
}

static int pipe_submit(tp_ctx* ctx, const tp_srs* srs, const Fr* const* scalars, int batch, size_t len) {
  MsmPipe* p = nullptr;
  TP_TRY(pipe_get(ctx, &p));
  if (batch <= 0 || batch > MSM_MAX_BATCH) return fail(ctx, TP_ERR_INVALID_ARG, "msm: bad batch size");
  if (p->results + batch > MSM_MAX_BATCH) return fail(ctx, TP_ERR_INVALID_ARG, "msm: too many results queued");
  if (len >= ((size_t)1 << 27)) return fail(ctx, TP_ERR_INVALID_ARG, "msm: more than 2^27 points per call");
  const unsigned world = ctx->world > 1 ? (unsigned)ctx->world : 1u;
  const MsmPlan pl = msm_plan(srs, world);
  if ((size_t)pl.nwin * len * batch >= ((size_t)1 << 31) || (size_t)pl.nsets * pl.nbuck * batch >= ((size_t)1 << 30)) {
    if (batch == 1) return fail(ctx, TP_ERR_INVALID_ARG, "msm: too many window entries");
    const int half = batch / 2;  // split the batch until the entry count fits 31 bits
    TP_TRY(pipe_submit(ctx, srs, scalars, half, len));
    return pipe_submit(ctx, srs, scalars + half, batch - half, len);
  }
  if (p->jobs.empty()) {   // first job of a batch fixes the mode
    p->overlap = msm_pipe_overlaps(ctx, len);
    if (p->overlap) TP_TRY(pipe_streams(ctx, p));
    p->win_used = 0;
    p->results = 0;
    if (!ctx->msm_winsums.p) TP_TRY(ensure(ctx, ctx->msm_winsums, ctx->pinned_cap));
  }
  MsmJob j;
  // one stream: a job has left its lane's buffers behind (in stream order) by the time the next one is queued, so
  // lane 0 serves them all -- the other lanes are only ever allocated by an overlapped batch
  j.lane = p->overlap ? p->next_lane : 0;
  if (p->overlap) p->next_lane = (p->next_lane + 1) % MSM_LANES;
  j.batch = batch;
  j.len = len;
  j.srs = srs;
  j.pl = pl;
  j.nsets_total = pl.nsets * (unsigned)batch;
  j.nkeys = (size_t)j.nsets_total * pl.nbuck;
  j.lazy = ctx->msm_fq_lazy != 0;
  j.first_result = p->results;
  p->results += batch;
  job_plan_reduce(ctx, j);
  j.win_off = p->win_used;
  p->win_used += (size_t)j.nsets_total * j.total_masks;
  // sharded, the host reads [slots 1.. summed over ranks | P of every rank] per set: world - 1 slots more than a rank writes
  size_t host_slots = 0;
  for (auto& q : p->jobs) host_slots += (size_t)q.nsets_total * (q.total_masks - 1 + world);
  j.host_off = world > 1 ? host_slots : j.win_off;
  host_slots += (size_t)j.nsets_total * (j.total_masks - 1 + world);
  if (p->win_used * sizeof(G1Xyzz) > ctx->msm_winsums.cap || host_slots * sizeof(G1Xyzz) > ctx->pinned_cap)
    return fail(ctx, TP_ERR_INVALID_ARG, "msm: staging buffer too small");
  if (len == 0) {
    j.empty = true;
    j.reduce_queued = true;
    p->jobs.push_back(j);
    return TP_OK;
  }
  MsmLane& ln = p->lane[j.lane];
  if (p->overlap) {
    // the scalars are final on the context's stream; the lane's buffers are free once its previous job has finished
    TP_CUDA_OK(ctx, cudaEventRecord(p->ev_in, ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamWaitEvent(p->s_sort, p->ev_in, 0));
    if (ln.busy) TP_CUDA_OK(ctx, cudaStreamWaitEvent(p->s_sort, ln.ev_done, 0));
  }
  TP_TRY(job_sort(ctx, p, j, scalars));
  if (p->overlap) TP_CUDA_OK(ctx, cudaEventSynchronize(ln.ev_sorted));
  else TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  j.m_total = p->counts[2 * j.lane];
  j.max_bucket = p->counts[2 * j.lane + 1];
  if (j.m_total == 0 && world == 1) {   // all scalars zero (a sharded rank still takes part in the exchange)
    j.empty = true;
    j.reduce_queued = true;
    p->jobs.push_back(j);
    return TP_OK;
  }
  TP_TRY(job_accumulate(ctx, p, j));
  ln.busy = p->overlap;
  // the reduction of the job before this one goes behind this job's accumulation (see the timeline above)
  if (p->overlap) {
    for (auto& q : p->jobs)
      if (!q.reduce_queued) TP_TRY(job_reduce(ctx, p, q));
  } else {
    TP_TRY(job_reduce(ctx, p, j));
  }
  p->jobs.push_back(j);
  return TP_OK;
}

static int pipe_finish(tp_ctx* ctx, tph::HG1* results, int count) {
  MsmPipe* p = ctx->msm_pipe;
  if (!p || p->results != count) return fail(ctx, TP_ERR_INVALID_ARG, "msm: finish does not match what was submitted");
  for (int b = 0; b < count; b++) results[b] = tph::HG1::identity();
  const unsigned world = ctx->world > 1 ? (unsigned)ctx->world : 1u;
  for (auto& q : p->jobs)
    if (!q.reduce_queued) TP_TRY(job_reduce(ctx, p, q));
  bool any = false;
  for (auto& q : p->jobs) any = any || !q.empty;
  if (any) {
    StreamSwap sw(ctx, pipe_tail_stream(ctx, p));
    // Sharded: the ranks' reduction outputs meet on the device -- one all-gather on the stream for the whole batch, one
    // combine kernel per job -- and the host reads back one buffer, as on a single GPU.
    const G1Xyzz* final_dev = (const G1Xyzz*)ctx->msm_winsums.p;
    size_t final_slots = p->win_used;
    if (world > 1) {
      ProfScope prof(ctx, TP_PHASE_MSM_REDUCE);
      const size_t per_rank = p->win_used * sizeof(G1Xyzz);
      size_t host_slots = 0;
      for (auto& q : p->jobs) host_slots += (size_t)q.nsets_total * (q.total_masks - 1 + world);
      TP_TRY(ensure_idle(ctx, ctx->msm_gather, per_rank * world + host_slots * sizeof(G1Xyzz)));
      G1Xyzz* gathered = (G1Xyzz*)ctx->msm_gather.p;
      G1Xyzz* combined = gathered + (size_t)world * p->win_used;
      TP_TRY(comm_allgather(ctx, ctx->msm_winsums.p, gathered, per_rank));
      for (auto& q : p->jobs) {
        if (q.empty) continue;
        (q.lazy ? k_msm_combine<true> : k_msm_combine<false>)<<<q.nsets_total * q.total_masks, 32, 0, ctx->stream>>>(gathered + q.win_off, world, (unsigned)p->win_used,
                                                                             q.total_masks, combined + q.host_off);
        TP_LAUNCH(ctx, "k_msm_combine");
      }
      final_dev = combined;
      final_slots = host_slots;
    }
    TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->pinned, final_dev, final_slots * sizeof(G1Xyzz), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  }
  for (auto& l : p->lane) l.busy = false;   // the tail stream has seen every job's last kernel
  // serial tails on the host
  const uint8_t* ws = (const uint8_t*)ctx->pinned;
  auto raw_point = [&](size_t index) {
    const uint8_t* q = ws + index * 192;
    tph::HFq x, y, zz, zzz;
    memcpy(x.v, q, 48);
    memcpy(y.v, q + 48, 48);
    memcpy(zz.v, q + 96, 48);
    memcpy(zzz.v, q + 144, 48);
    return tph::g1_from_xyzz(x, y, zz, zzz);
  };
  // one bucket set's tail is ~40 dependent group operations of single-thread host arithmetic (~0.1 ms); the sets of a
  // batch are independent, so every result beyond the first gets its own thread
  auto tail = [&](const MsmJob* jp, int b) {
    const MsmJob& j = *jp;
    const MsmPlan& pl = j.pl;
    const unsigned width = world > 1 ? j.total_masks - 1 + world : j.total_masks;
    // slot >= 1 of a set (summed over ranks when sharded)
    auto point = [&](unsigned set, unsigned slot) { return raw_point(j.host_off + (size_t)set * width + (world > 1 ? slot - 1 : slot)); };
    tph::HG1 acc = tph::HG1::identity();
    for (int q = (int)pl.nsets - 1; q >= 0; q--) {
      if (q != (int)pl.nsets - 1)
        for (unsigned d = 0; d < pl.c * pl.levels; d++) acc = tph::g1_dbl(acc);
      unsigned set = (unsigned)b * pl.nsets + (unsigned)q;
      // F(X) = F(C) + cols * F(D), each from its bit sums (Horner from the top bit); X = the R array of the last
      // running-sum level, unwound level by level
      auto bits = [&](unsigned first_slot, unsigned nb) {
        tph::HG1 v = tph::HG1::identity();
        for (int k = (int)nb - 1; k >= 0; k--) {
          v = tph::g1_dbl(v);
          v = tph::g1_add(v, point(set, first_slot + (unsigned)k));
        }
        return v;
      };
      tph::HG1 f = bits(1, j.bD);
      for (unsigned d = 0; d < j.bC; d++) f = tph::g1_dbl(f);
      f = tph::g1_add(f, bits(1 + j.bD, j.bC));
      for (int l = j.nl; l >= 1; l--) {  // F(level l-1) = T_l + S_l * F(level l)
        for (unsigned d = 1; d < j.seg_level[l]; d <<= 1) f = tph::g1_dbl(f);
        f = tph::g1_add(f, point(set, 1 + j.bD + j.bC + (unsigned)(l - 1)));
      }
      if (world == 1) {
        f = tph::g1_add(f, raw_point(j.host_off + (size_t)set * width));   // V = F + P
      } else {
        // local bucket j of rank r is global bucket world * j + r, which counts (world * j + r + 1) times:
        // V = world * F(summed over ranks) + sum_r (r + 1) P_r, the latter by running sums
        tph::HG1 wf = tph::HG1::identity();
        for (int bit = 31 - __builtin_clz(world); bit >= 0; bit--) {
          wf = tph::g1_dbl(wf);
          if ((world >> bit) & 1) wf = tph::g1_add(wf, f);
        }
        tph::HG1 run = tph::HG1::identity(), pw = tph::HG1::identity();
        for (int r = (int)world - 1; r >= 0; r--) {
          run = tph::g1_add(run, raw_point(j.host_off + (size_t)set * width + (j.total_masks - 1) + (unsigned)r));
          pw = tph::g1_add(pw, run);
        }
        f = tph::g1_add(wf, pw);
      }
      acc = tph::g1_add(acc, f);
    }
    results[j.first_result + b] = acc;
  };
  std::vector<std::pair<const MsmJob*, int>> work;
  for (auto& q : p->jobs)
    if (!q.empty)
      for (int b = 0; b < q.batch; b++) work.push_back({&q, b});
  std::vector<std::future<void>> others;
  size_t w_next = 1;
  try {
    for (; w_next < work.size(); w_next++) others.push_back(std::async(std::launch::async, tail, work[w_next].first, work[w_next].second));
  } catch (const std::system_error&) {  // no more threads to be had: the rest runs here
  }
  if (!work.empty()) tail(work[0].first, work[0].second);
  for (size_t w = w_next; w < work.size(); w++) tail(work[w].first, work[w].second);
  for (auto& f : others) f.get();
  p->jobs.clear();
  p->win_used = 0;
  p->results = 0;
  return TP_OK;
}

int msm_pipe_submit(tp_ctx* ctx, const tp_srs* srs, const Fr* const* scalars_dev, int batch, size_t len) {
  if (len > srs->len) return fail(ctx, TP_ERR_SRS_TOO_SHORT, "commit: polynomial longer than the SRS");
  if (ctx->world > 1 && !comm_ready(ctx)) return fail(ctx, TP_ERR_COLLECTIVE, "msm: sharded context without a communicator");
  MsmPipe* p = nullptr;
  TP_TRY(pipe_get(ctx, &p));
  const bool first = p->jobs.empty();
  const bool overlap = first ? msm_pipe_overlaps(ctx, len) : p->overlap;
  int rc;
  if (overlap) {   // the work spreads over the pipe's streams: the total runs from here to the end of finish
    if (first && ctx->prof && !p->total) p->total = new ProfScope(ctx, TP_PHASE_MSM_TOTAL);
    rc = pipe_submit(ctx, srs, scalars_dev, batch, len);
  } else {
    ProfScope prof(ctx, TP_PHASE_MSM_TOTAL);
    rc = pipe_submit(ctx, srs, scalars_dev, batch, len);
  }
  if (rc != TP_OK) pipe_abort(ctx);
  return rc;
}
int msm_pipe_finish(tp_ctx* ctx, uint8_t (*out)[TP_G1_BYTES], int count) {
  if (count < 0 || count > MSM_MAX_BATCH) return fail(ctx, TP_ERR_INVALID_ARG, "msm: bad result count");
  tph::HG1 res[MSM_MAX_BATCH];
  MsmPipe* p = ctx->msm_pipe;
  int rc;
  if (p && p->total) {
    rc = pipe_finish(ctx, res, count);   // ends with the host waiting for the tail stream: everything has run
    delete p->total;
    p->total = nullptr;
  } else {
    ProfScope prof(ctx, TP_PHASE_MSM_TOTAL);
    rc = pipe_finish(ctx, res, count);
  }
  if (rc != TP_OK) {
    pipe_abort(ctx);
    return rc;
  }
  encode_g1_batch(res, out, count);
  return TP_OK;
}

// Sub-batch sizes of a batch run in one call: at most three jobs, the first the smallest (its sort is the one nothing
// covers).  TP_MSM_PIPE_PARTS=a,b,c overrides for sweeps (missing or short: equal parts).
static int msm_split(int batch, int parts[MSM_LANES]) {
  static const char* env = getenv("TP_MSM_PIPE_PARTS");
  int n = batch < MSM_LANES ? batch : MSM_LANES;
  for (int i = 0; i < n; i++) parts[i] = batch / n + (i >= n - batch % n ? 1 : 0);
  if (env && *env) {
    int v[MSM_LANES] = {0, 0, 0}, sum = 0, cnt = 0;
    const char* s = env;
    while (*s && cnt < MSM_LANES) {
      v[cnt] = (int)strtol(s, (char**)&s, 10);
      sum += v[cnt] > 0 ? v[cnt] : 0;
      if (v[cnt] > 0) cnt++;
      if (*s == ',') s++;
      else break;
    }
    if (sum == batch && cnt > 0) {
      for (int i = 0; i < cnt; i++) parts[i] = v[i];
      n = cnt;
    }
  }
  return n;
}

// `batch` MSMs over the first `len` bases: out[b] = sum_i scalars[b][i] * srs[i].  Overlapped, the batch is cut into
// sub-batches (see "pipeline"); otherwise all scalar vectors share one sort / accumulate / merge / reduce pass (bucket
// set index = b * nsets + q), which amortises the latency-bound reduction tail and the launch overhead.  On a sharded
// context (world > 1) this rank handles the buckets it owns, the ranks' reduction outputs are all-gathered and combined
// on the device (comm.cu, k_msm_combine) and every rank returns the complete sums.
int msm_batch_dev(tp_ctx* ctx, const tp_srs* srs, const Fr* const* scalars_dev, int batch, size_t len,
                  uint8_t (*out)[TP_G1_BYTES]) {
  if (batch <= 0 || batch > MSM_MAX_BATCH) return fail(ctx, TP_ERR_INVALID_ARG, "msm: bad batch size");
  if (ctx->msm_pipe && !ctx->msm_pipe->jobs.empty()) return fail(ctx, TP_ERR_INVALID_ARG, "msm: a submitted batch is still open");
  if (msm_pipe_overlaps(ctx, len) && batch > 1) {
    int parts[MSM_LANES];
    const int n = msm_split(batch, parts);
    int at = 0;
    for (int i = 0; i < n; i++) {
      TP_TRY(msm_pipe_submit(ctx, srs, scalars_dev + at, parts[i], len));
      at += parts[i];
    }
  } else {
    TP_TRY(msm_pipe_submit(ctx, srs, scalars_dev, batch, len));
  }
  return msm_pipe_finish(ctx, out, batch);
}

int msm_dev(tp_ctx* ctx, const tp_srs* srs, const Fr* scalars_dev, size_t len, uint8_t out[TP_G1_BYTES]) {
  const Fr* one[1] = {scalars_dev};
  return msm_batch_dev(ctx, srs, one, 1, len, (uint8_t(*)[TP_G1_BYTES])out);
}

}  // namespace tp
