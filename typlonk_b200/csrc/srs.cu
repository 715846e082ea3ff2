// SRS generation on the device: [G, tau G, tau^2 G, ...] (kzg/src/srs.rs:15-24, which the
// reference computes as `length` serial double-and-add multiplications).  Here: every thread
// takes 8 consecutive powers of tau (one pow, then a multiply chain), multiplies the generator
// by each with a fixed-base table of 32 windows x 255 affine multiples (32 mixed additions per
// point, no doublings), and normalises its 8 results to affine with one shared inversion.  A ceremony contribution
// (k_srs_contribute, srs_ceremony.cu) rescales an existing SRS by the powers of a new secret in the same shape.
#include "common.cuh"

namespace tp {

#define SRS_PER 8
#define FB_WINDOWS 32
#define FB_ENTRIES 255

static const uint64_t G1_GEN_X[6] = {0xfb3af00adb22c6bbull, 0x6c55e83ff97a1aefull, 0xa14e3a3f171bac58ull,
                                     0xc3688c4f9774b905ull, 0x2695638c4fa9ac0full, 0x17f1d3a73197d794ull};
static const uint64_t G1_GEN_Y[6] = {0x0caa232946c5e7e1ull, 0xd03cc744a2888ae4ull, 0x00db18cb2c04b3edull,
                                     0xfcf5e095d5d00af6ull, 0xa09e30ed741d8ae4ull, 0x08b3f481e3aaa0f1ull};

tph::HG1 host_generator() {
  return tph::g1_from_affine(tph::HFq::to_mont(G1_GEN_X), tph::HFq::to_mont(G1_GEN_Y));
}

static int build_fixed_base(tp_ctx* ctx) {
  if (ctx->fixed_base) return TP_OK;
  const size_t count = (size_t)FB_WINDOWS * FB_ENTRIES;
  std::vector<tph::HG1> pts(count);
  tph::HG1 base = host_generator();
  for (int j = 0; j < FB_WINDOWS; j++) {
    tph::HG1 acc = base;
    for (int d = 0; d < FB_ENTRIES; d++) {
      pts[(size_t)j * FB_ENTRIES + d] = acc;
      acc = tph::g1_add(acc, base);
    }
    base = acc;  // 256 * base
  }
  // batch affine conversion
  std::vector<tph::HFq> pre(count);
  tph::HFq acc = tph::HFq::one();
  for (size_t i = 0; i < count; i++) {
    pre[i] = acc;
    acc = acc * pts[i].z;
  }
  tph::HFq inv = acc.inv();
  std::vector<uint8_t> packed(count * 96);
  for (size_t i = count; i-- > 0;) {
    tph::HFq zi = inv * pre[i];
    inv = inv * pts[i].z;
    tph::HFq zi2 = zi.sqr();
    tph::HFq x = pts[i].x * zi2, y = pts[i].y * zi2 * zi;
    memcpy(&packed[i * 96], x.v, 48);
    memcpy(&packed[i * 96 + 48], y.v, 48);
  }
  TP_CUDA_OK(ctx, cudaMalloc(&ctx->fixed_base, count * 96));
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->fixed_base, packed.data(), count * 96, cudaMemcpyHostToDevice, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return TP_OK;
}

// The tail every kernel below shares: a thread's `cnt` XYZZ results to packed affine records out[0 .. cnt), with one
// shared inversion of the product of their zz * zzz (the identity stays the all-zero record).
__device__ __forceinline__ void store_affine(const G1Xyzz (&pts)[SRS_PER], int cnt, G1Affine* __restrict__ out) {
  Fq pre[SRS_PER];
  Fq acc = fq_one();
  for (int i = 0; i < cnt; i++) {
    pre[i] = acc;
    Fq d = xyzz_is_identity(pts[i]) ? fq_one() : fq_mul(pts[i].zz, pts[i].zzz);
    acc = fq_mul(acc, d);
  }
  Fq inv = fq_inv(acc);
  for (int i = cnt - 1; i >= 0; i--) {
    G1Affine r;
    if (xyzz_is_identity(pts[i])) {
      r.x = fq_zero();
      r.y = fq_zero();
    } else {
      Fq d = fq_mul(pts[i].zz, pts[i].zzz);
      Fq di = fq_mul(inv, pre[i]);  // 1 / (zz zzz)
      inv = fq_mul(inv, d);
      r.x = fq_mul(pts[i].x, fq_mul(di, pts[i].zzz));  // X / ZZ
      r.y = fq_mul(pts[i].y, fq_mul(di, pts[i].zz));   // Y / ZZZ
    }
    fq_store(&out[i].x, r.x);
    fq_store(&out[i].y, r.y);
  }
}

__global__ void __launch_bounds__(64) k_srs_generate(const G1Affine* __restrict__ table, Fr tau, size_t len,
                                                     G1Affine* __restrict__ out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * SRS_PER;
  if (lo >= len) return;
  int cnt = (int)(lo + SRS_PER < len ? SRS_PER : len - lo);
  G1Xyzz pts[SRS_PER];
  Fr power = fr_pow_u64(tau, (unsigned long long)lo);
  for (int i = 0; i < cnt; i++) {
    Fr s = fr_from_mont(power);
    G1Xyzz acc = xyzz_identity();
    for (int j = 0; j < FB_WINDOWS; j++) {
      unsigned d = (s.v[j >> 2] >> ((j & 3) * 8)) & 0xffu;
      if (d) {
        G1Affine p = affine_load(table + (size_t)j * FB_ENTRIES + (d - 1));
        xyzz_madd(acc, p, false);
      }
    }
    pts[i] = acc;
    power = fr_mul(power, tau);
  }
  store_affine(pts, cnt, out + lo);
}

// Fixed-base window tables: level k+1 = 2^c * level k.  Every thread doubles SRS_PER consecutive
// points c times in XYZZ and normalises them with one shared inversion.
__global__ void __launch_bounds__(64) k_srs_next_level(const G1Affine* __restrict__ in, size_t len, unsigned c,
                                                       G1Affine* __restrict__ out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * SRS_PER;
  if (lo >= len) return;
  int cnt = (int)(lo + SRS_PER < len ? SRS_PER : len - lo);
  G1Xyzz pts[SRS_PER];
  for (int i = 0; i < cnt; i++) {
    G1Affine p = affine_load(in + lo + i);
    G1Xyzz acc = xyzz_identity();
    if (!affine_is_identity(p)) {
      xyzz_mdbl(acc, p);
      for (unsigned d = 1; d < c; d++) xyzz_dbl(acc);
    }
    pts[i] = acc;
  }
  store_affine(pts, cnt, out + lo);
}

// One powers-of-tau contribution: out[i] = [s^i] in[i].  Every thread takes SRS_PER consecutive points (one pow, then a
// multiply chain for the scalars), runs an MSB-first XYZZ double-and-add from each affine point -- the ladder of
// g1_in_subgroup, ~254 doublings and ~127 mixed additions for a random scalar -- and normalises its results with one
// shared inversion.  An input identity stays the identity; s^0 = 1 leaves in[0] as it is.
__global__ void __launch_bounds__(64) k_srs_contribute(const G1Affine* __restrict__ in, Fr s, size_t len,
                                                       G1Affine* __restrict__ out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * SRS_PER;
  if (lo >= len) return;
  int cnt = (int)(lo + SRS_PER < len ? SRS_PER : len - lo);
  G1Xyzz pts[SRS_PER];
  Fr power = fr_pow_u64(s, (unsigned long long)lo);
  for (int i = 0; i < cnt; i++) {
    Fr k = fr_from_mont(power);
    power = fr_mul(power, s);
    G1Affine p = affine_load(in + lo + i);
    G1Xyzz acc = xyzz_identity();
    int top = 7;
    while (top >= 0 && k.v[top] == 0) top--;
    if (top >= 0 && !affine_is_identity(p)) {
      acc.x = p.x;
      acc.y = p.y;
      acc.zz = fq_one();
      acc.zzz = fq_one();
      for (int bit = top * 32 + 30 - __clz(k.v[top]); bit >= 0; bit--) {   // below the leading one
        xyzz_dbl(acc);
        if ((k.v[bit >> 5] >> (bit & 31)) & 1) xyzz_madd(acc, p, false);
      }
    }
    pts[i] = acc;
  }
  store_affine(pts, cnt, out + lo);
}

int srs_build_levels_dev(tp_ctx* ctx, tp_srs* srs) {
  if (srs->len == 0) return TP_OK;
  size_t nth = (srs->len + SRS_PER - 1) / SRS_PER;
  for (unsigned k = 1; k < srs->levels; k++) {
    k_srs_next_level<<<(unsigned)((nth + 63) / 64), 64, 0, ctx->stream>>>(srs->g1 + (size_t)(k - 1) * srs->len, srs->len,
                                                                          srs->c, srs->g1 + (size_t)k * srs->len);
    TP_LAUNCH(ctx, "k_srs_next_level");
  }
  return TP_OK;
}

int srs_generate_dev(tp_ctx* ctx, const tph::HFr& tau, size_t len, G1Affine* out) {
  TP_TRY(build_fixed_base(ctx));
  size_t nth = (len + SRS_PER - 1) / SRS_PER;
  k_srs_generate<<<(unsigned)((nth + 63) / 64), 64, 0, ctx->stream>>>((const G1Affine*)ctx->fixed_base, to_dev(tau), len,
                                                                    out);
  TP_LAUNCH(ctx, "k_srs_generate");
  return TP_OK;
}

int srs_contribute_dev(tp_ctx* ctx, const G1Affine* in, const tph::HFr& s, size_t len, G1Affine* out) {
  if (len == 0) return TP_OK;
  size_t nth = (len + SRS_PER - 1) / SRS_PER;
  k_srs_contribute<<<(unsigned)((nth + 63) / 64), 64, 0, ctx->stream>>>(in, to_dev(s), len, out);
  TP_LAUNCH(ctx, "k_srs_contribute");
  return TP_OK;
}

}  // namespace tp
