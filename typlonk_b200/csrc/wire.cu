// Wire formats (SURVEY.md 8 f4, App. A.6): a proof and an SRS as bytes, in the encoding ark-serialize 0.3 gives the
// reference's own types -- the same one its Fiat-Shamir transcript already uses for G1 (plonk/src/proof/challenges.rs:17-22):
//   Fr  32 B little-endian canonical integer
//   G1  96 B uncompressed: x | y, 48 B little-endian canonical each; bit 6 of the last byte = point at infinity
//       (stored as x = 0, y = 1); bit 7 is the y-sign flag of the COMPRESSED form and must be clear here
//   G2  192 B uncompressed: x.c0 | x.c1 | y.c0 | y.c1, same flag convention
//   Vec u64 little-endian length, then the items
// Proof (plonk/src/proof.rs:85-95)  = the 1472-byte block tp_prove writes | Vec<Fr> public inputs.
// SRS   (kzg/src/srs.rs:8-14)       = Vec<G1> | G2 | tau G2.
// The reference derives neither Serialize nor Deserialize for these types, so the framing is ours; every item inside
// it is what arkworks would write.  Proofs are small and handled on the host; the SRS (100 MB at 2^20) is converted
// out of / into Montgomery form and validated (canonical, on the curve, optionally in the prime-order subgroup) on
// the device, one point per thread.
#include "circuit.h"
#include "ec.cuh"
#include "pairing.h"

using namespace tp;
using namespace tph;

namespace tp {

__device__ __forceinline__ bool fq_lt_mod(const Fq& a) {
  const uint32_t m[12] = TP_FQ_MOD;
  for (int i = 11; i >= 0; i--) {
    if (a.v[i] < m[i]) return true;
    if (a.v[i] > m[i]) return false;
  }
  return false;
}
__device__ __forceinline__ Fq fq_to_mont(const Fq& a) {
  const uint32_t c[12] = TP_FQ_R2;
  Fq r2;
#pragma unroll
  for (int i = 0; i < 12; i++) r2.v[i] = c[i];
  return fq_mul(a, r2);
}
__device__ __forceinline__ Fq fq_from_mont(const Fq& a) {
  Fq o = fq_zero();
  o.v[0] = 1;
  return fq_mul(a, o);
}

// Montgomery SRS records -> wire records.  96 B per thread as six 16-byte stores.
__global__ void __launch_bounds__(128) k_g1_to_wire(const G1Affine* __restrict__ in, size_t len, uint4* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    G1Affine p = affine_load(in + i);
    Fq x, y;
    if (affine_is_identity(p)) {
      x = fq_zero();
      y = fq_zero();
      y.v[0] = 1;
      y.v[11] |= 0x40000000u;  // bit 6 of byte 95
    } else {
      x = fq_from_mont(p.x);
      y = fq_from_mont(p.y);
    }
    uint4* o = out + i * 6;
    o[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    o[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
    o[2] = make_uint4(x.v[8], x.v[9], x.v[10], x.v[11]);
    o[3] = make_uint4(y.v[0], y.v[1], y.v[2], y.v[3]);
    o[4] = make_uint4(y.v[4], y.v[5], y.v[6], y.v[7]);
    o[5] = make_uint4(y.v[8], y.v[9], y.v[10], y.v[11]);
  }
}

// Wire records -> Montgomery SRS records, validated.  check: 0 = canonical encoding only (deserialize_unchecked),
// 1 = + on the curve, 2 = + in the prime-order subgroup (what ark-ec's checked deserialisation enforces).
// bad[0] counts rejected records, bad[1] keeps the lowest rejected index + 1.
__global__ void __launch_bounds__(128) k_g1_from_wire(const uint4* __restrict__ in, size_t len, int check,
                                                      G1Affine* __restrict__ out, unsigned long long* __restrict__ bad) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    const uint4* s = in + i * 6;
    Fq x, y;
    uint4 q;
    q = s[0]; x.v[0] = q.x; x.v[1] = q.y; x.v[2] = q.z; x.v[3] = q.w;
    q = s[1]; x.v[4] = q.x; x.v[5] = q.y; x.v[6] = q.z; x.v[7] = q.w;
    q = s[2]; x.v[8] = q.x; x.v[9] = q.y; x.v[10] = q.z; x.v[11] = q.w;
    q = s[3]; y.v[0] = q.x; y.v[1] = q.y; y.v[2] = q.z; y.v[3] = q.w;
    q = s[4]; y.v[4] = q.x; y.v[5] = q.y; y.v[6] = q.z; y.v[7] = q.w;
    q = s[5]; y.v[8] = q.x; y.v[9] = q.y; y.v[10] = q.z; y.v[11] = q.w;
    const uint32_t flags = y.v[11] >> 30;
    y.v[11] &= 0x3fffffffu;
    bool ok = !(flags & 2) && fq_lt_mod(x) && fq_lt_mod(y);
    G1Affine p;
    if (flags & 1) {  // infinity: canonical only as (x, y) = (0, 1); the device SRS keeps it as the all-zero record
      bool canon = x.v[0] == 0 && y.v[0] == 1;
#pragma unroll
      for (int k = 1; k < 12; k++) canon = canon && x.v[k] == 0 && y.v[k] == 0;
      ok = ok && canon;
      p.x = fq_zero();
      p.y = fq_zero();
    } else {
      p.x = fq_to_mont(x);
      p.y = fq_to_mont(y);
      if (ok && check >= 1) {
        Fq four = fq_dbl(fq_dbl(fq_one()));
        ok = fq_eq(fq_sqr(p.y), fq_add(fq_mul(fq_sqr(p.x), p.x), four));
      }
      if (ok && check >= 2) ok = g1_in_subgroup(p);
    }
    fq_store(&out[i].x, p.x);
    fq_store(&out[i].y, p.y);
    if (!ok) {
      atomicAdd(bad, 1ull);
      atomicMin(bad + 1, (unsigned long long)i + 1);
    }
  }
}

static unsigned wire_grid(tp_ctx* ctx, size_t len) {
  size_t blocks = (len + 127) / 128;
  size_t cap = (size_t)ctx->sm_count * 16;
  return (unsigned)(blocks < cap ? (blocks ? blocks : 1) : cap);
}

int g1_to_wire_dev(tp_ctx* ctx, const G1Affine* in, size_t len, void* out_dev) {
  if (!len) return TP_OK;
  k_g1_to_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>(in, len, (uint4*)out_dev);
  TP_LAUNCH(ctx, "k_g1_to_wire");
  return TP_OK;
}

int g1_from_wire_dev(tp_ctx* ctx, const void* in_dev, size_t len, int check, G1Affine* out, size_t* rejected,
                     size_t* first_rejected) {
  *rejected = 0;
  *first_rejected = 0;
  if (!len) return TP_OK;
  TP_TRY(ensure(ctx, ctx->flag, 16));
  unsigned long long init[2] = {0, ~0ull}, got[2];
  TP_CUDA_OK(ctx, cudaMemcpyAsync(ctx->flag.p, init, 16, cudaMemcpyHostToDevice, ctx->stream));
  k_g1_from_wire<<<wire_grid(ctx, len), 128, 0, ctx->stream>>>((const uint4*)in_dev, len, check, out,
                                                                (unsigned long long*)ctx->flag.p);
  TP_LAUNCH(ctx, "k_g1_from_wire");
  TP_CUDA_OK(ctx, cudaMemcpyAsync(got, ctx->flag.p, 16, cudaMemcpyDeviceToHost, ctx->stream));
  TP_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  *rejected = (size_t)got[0];
  *first_rejected = got[0] ? (size_t)(got[1] - 1) : 0;
  return TP_OK;
}

// ---- host side: single items ---------------------------------------------------------------------------------------
static void fq_to_wire(const HFq& a, uint8_t out[48]) {
  HFq c = a.from_mont();
  memcpy(out, c.v, 48);
}
static bool fq_from_wire(const uint8_t in[48], uint8_t flag_mask, HFq* out, uint8_t* flags) {
  uint64_t v[6];
  memcpy(v, in, 48);
  if (flags) *flags = (uint8_t)(v[5] >> 56) & flag_mask;
  v[5] &= ~((uint64_t)flag_mask << 56);
  if (ge<6>(v, FQ_PARAMS.mod)) return false;
  *out = HFq::to_mont(v);
  return true;
}

void g2_to_wire(const G2Aff& p, uint8_t out[TP_WIRE_G2_BYTES]) {
  if (p.inf) {
    memset(out, 0, TP_WIRE_G2_BYTES);
    out[96] = 1;
    out[191] |= 0x40;
    return;
  }
  fq_to_wire(p.x.a, out);
  fq_to_wire(p.x.b, out + 48);
  fq_to_wire(p.y.a, out + 96);
  fq_to_wire(p.y.b, out + 144);
}
bool g2_from_wire(const uint8_t in[TP_WIRE_G2_BYTES], int check, G2Aff* out) {
  uint8_t flags = 0;
  G2Aff p;
  p.inf = false;
  bool ok = fq_from_wire(in, 0, &p.x.a, nullptr) && fq_from_wire(in + 48, 0, &p.x.b, nullptr) &&
            fq_from_wire(in + 96, 0, &p.y.a, nullptr) && fq_from_wire(in + 144, 0xc0, &p.y.b, &flags);
  if (!ok || (flags & 0x80)) return false;
  if (flags & 0x40) {  // infinity is canonical only as (x, y) = (0, 1)
    if (!(p.x == Fq2::zero()) || !(p.y == Fq2::one())) return false;
    *out = {Fq2::zero(), Fq2::one(), true};
    return true;
  }
  if (check >= 1 && !g2_on_curve(p)) return false;
  if (check >= 2 && !g2_mul(p, FR_PARAMS.mod, 4).inf) return false;
  *out = p;
  return true;
}

static bool g1_wire_valid(const uint8_t in[TP_WIRE_G1_BYTES]) {
  uint8_t flags = 0;
  G1Aff p;
  p.inf = false;
  if (!fq_from_wire(in, 0, &p.x, nullptr) || !fq_from_wire(in + 48, 0xc0, &p.y, &flags)) return false;
  if (flags & 0x80) return false;
  if (flags & 0x40) return p.x == HFq::zero() && p.y == HFq::one();  // infinity is canonical only as (0, 1)
  return g1aff_on_curve(p);
}

}  // namespace tp

// ---- the proof -----------------------------------------------------------------------------------------------------
// proof.rs:85-95 in the order tp_prove writes it: G = a G1 point, F = a scalar.
static const char kProofLayout[] = "GGF" "GGF" "GGF" "GGF" "GF" "F" "GGG" "GF";

extern "C" {

int tp_proof_encoded_size(size_t n_public, size_t* bytes) {
  if (!bytes) return TP_ERR_INVALID_ARG;
  *bytes = TP_PROOF_FIXED_BYTES + 8 + 32 * n_public;
  return TP_OK;
}

int tp_proof_encode(const uint8_t* fixed, const uint64_t* public_inputs, size_t n_public, uint8_t* out, size_t cap,
                    size_t* written) {
  if (!fixed || !out || (n_public && !public_inputs)) return TP_ERR_INVALID_ARG;
  const size_t need = TP_PROOF_FIXED_BYTES + 8 + 32 * n_public;
  if (written) *written = need;
  if (cap < need) return TP_ERR_BUFFER_TOO_SMALL;
  memcpy(out, fixed, TP_PROOF_FIXED_BYTES);
  uint64_t n64 = n_public;
  memcpy(out + TP_PROOF_FIXED_BYTES, &n64, 8);
  uint8_t* o = out + TP_PROOF_FIXED_BYTES + 8;
  for (size_t i = 0; i < n_public; i++, o += 32) {
    HFr v;
    memcpy(v.v, public_inputs + 4 * i, 32);
    if (ge<4>(v.v, FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
    HFr c = v.from_mont();
    memcpy(o, c.v, 32);
  }
  return TP_OK;
}

// ark-serialize's CHECKED deserialisation also verifies [r]P = 0 for every point; tp_proof_decode stops at "on the
// curve" (the reference's transcript uses the unchecked form).  This is the additional check, on the host: 13 scalar
// multiplications by r.
int tp_proof_points_in_subgroup(const uint8_t* fixed, size_t len, int* ok) {
  if (!fixed || !ok || len < TP_PROOF_FIXED_BYTES) return TP_ERR_INVALID_ARG;
  *ok = 0;
  const uint8_t* p = fixed;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k != 'G') {
      p += 32;
      continue;
    }
    if (!tp::g1_wire_valid(p)) return TP_ERR_MALFORMED;
    uint8_t flags = 0;
    G1Aff a;
    a.inf = false;
    tp::fq_from_wire(p, 0, &a.x, nullptr);
    tp::fq_from_wire(p + 48, 0xc0, &a.y, &flags);
    if (!(flags & 0x40)) {
      HG1 m = g1_mul_u64limbs(g1_from_affine(a.x, a.y), FR_PARAMS.mod, 4);
      if (!m.is_identity()) return TP_OK;   // *ok stays 0
    }
    p += TP_WIRE_G1_BYTES;
  }
  *ok = 1;
  return TP_OK;
}

int tp_proof_decode(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_FIXED_BYTES],
                    uint64_t* public_inputs_out, size_t cap_public, size_t* n_public) {
  if (!bytes || !n_public) return TP_ERR_INVALID_ARG;
  if (len < TP_PROOF_FIXED_BYTES + 8) return TP_ERR_MALFORMED;
  uint64_t n64;
  memcpy(&n64, bytes + TP_PROOF_FIXED_BYTES, 8);
  if (n64 > (len - TP_PROOF_FIXED_BYTES - 8) / 32 || len != TP_PROOF_FIXED_BYTES + 8 + 32 * (size_t)n64)
    return TP_ERR_MALFORMED;
  const uint8_t* p = bytes;
  for (const char* k = kProofLayout; *k; k++) {
    if (*k == 'G') {
      if (!tp::g1_wire_valid(p)) return TP_ERR_MALFORMED;
      p += TP_WIRE_G1_BYTES;
    } else {
      uint64_t v[4];
      memcpy(v, p, 32);
      if (ge<4>(v, FR_PARAMS.mod)) return TP_ERR_MALFORMED;
      p += 32;
    }
  }
  p += 8;
  for (size_t i = 0; i < n64; i++) {
    uint64_t v[4];
    memcpy(v, p + 32 * i, 32);
    if (ge<4>(v, FR_PARAMS.mod)) return TP_ERR_MALFORMED;
  }
  *n_public = (size_t)n64;
  if (public_inputs_out) {
    if (cap_public < n64) return TP_ERR_BUFFER_TOO_SMALL;
    for (size_t i = 0; i < n64; i++) {
      uint64_t v[4];
      memcpy(v, p + 32 * i, 32);
      HFr m = HFr::to_mont(v);
      memcpy(public_inputs_out + 4 * i, m.v, 32);
    }
  }
  if (fixed_out) memcpy(fixed_out, bytes, TP_PROOF_FIXED_BYTES);
  return TP_OK;
}

}  // extern "C"

// ---- the SRS -------------------------------------------------------------------------------------------------------
extern "C" {

int tp_srs_serialized_size(const tp_srs* srs, size_t* bytes) {
  if (!srs || !bytes) return TP_ERR_INVALID_ARG;
  *bytes = 8 + srs->len * TP_WIRE_G1_BYTES + 2 * TP_WIRE_G2_BYTES;
  return TP_OK;
}

int tp_srs_serialize(tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written) {
  if (!ctx || !srs || !out) return TP_ERR_INVALID_ARG;
  if (!ctx->children.empty())   // device group: rank 0's copy
    return group_run(ctx, [&](tp_ctx* c, int r) { return r == 0 ? tp_srs_serialize(c, srs->parts[0], out, cap, written) : TP_OK; });
  if (!srs->pairing) return fail(ctx, TP_ERR_INVALID_ARG, "srs_serialize: the SRS has no G2 points (tp_srs_set_g2)");
  const size_t need = 8 + srs->len * TP_WIRE_G1_BYTES + 2 * TP_WIRE_G2_BYTES;
  if (written) *written = need;
  if (cap < need) return fail(ctx, TP_ERR_BUFFER_TOO_SMALL, "srs_serialize: output buffer too small");
  uint64_t n64 = srs->len;
  memcpy(out, &n64, 8);
  if (srs->len) {
    void* stage = nullptr;
    TP_CUDA_OK(ctx, cudaMalloc(&stage, srs->len * TP_WIRE_G1_BYTES));
    int rc = g1_to_wire_dev(ctx, srs->g1, srs->len, stage);
    if (rc == TP_OK && (cudaMemcpyAsync(out + 8, stage, srs->len * TP_WIRE_G1_BYTES, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                        cudaStreamSynchronize(ctx->stream) != cudaSuccess))
      rc = fail(ctx, TP_ERR_CUDA, "srs_serialize: copy failed");
    cudaFree(stage);
    if (rc != TP_OK) return rc;
  }
  uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
  if (tp_srs_g2(srs, g2, g2s) != TP_OK) return fail(ctx, TP_ERR_INVALID_ARG, "srs_serialize: no G2 points");
  uint8_t* o = out + 8 + srs->len * TP_WIRE_G1_BYTES;
  g2_to_wire(g2_decode(g2), o);
  g2_to_wire(g2_decode(g2s), o + TP_WIRE_G2_BYTES);
  return TP_OK;
}

int tp_srs_deserialize(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out) {
  if (!ctx || !bytes || !out || check < 0 || check > 2) return TP_ERR_INVALID_ARG;
  if (!ctx->children.empty()) {   // device group: every rank decodes (and validates) its own copy
    tp_srs* front = new tp_srs();
    front->parts.assign(ctx->children.size(), nullptr);
    int rc = group_run(ctx, [&](tp_ctx* c, int r) { return tp_srs_deserialize(c, bytes, len, check, &front->parts[r]); });
    if (rc != TP_OK) {
      group_run(ctx, [&](tp_ctx* c, int r) { return tp_srs_destroy(c, front->parts[r]); });
      delete front;
      return rc;
    }
    front->len = front->parts[0]->len;
    *out = front;
    return TP_OK;
  }
  if (len < 8 + 2 * TP_WIRE_G2_BYTES) return fail(ctx, TP_ERR_MALFORMED, "srs_deserialize: truncated");
  uint64_t n64;
  memcpy(&n64, bytes, 8);
  const size_t body = len - 8 - 2 * TP_WIRE_G2_BYTES;
  if (n64 > body / TP_WIRE_G1_BYTES || body != (size_t)n64 * TP_WIRE_G1_BYTES)
    return fail(ctx, TP_ERR_MALFORMED, "srs_deserialize: length does not match the point count");
  const size_t n = (size_t)n64;
  G2Aff q, qs;
  const uint8_t* tail = bytes + 8 + n * TP_WIRE_G1_BYTES;
  if (!g2_from_wire(tail, check, &q) || !g2_from_wire(tail + TP_WIRE_G2_BYTES, check, &qs))
    return fail(ctx, TP_ERR_MALFORMED, "srs_deserialize: bad G2 point");
  tp_srs* s = nullptr;
  TP_TRY(srs_alloc(ctx, n, &s));
  int rc = TP_OK;
  size_t rejected = 0, first = 0;
  if (n) {
    void* stage = nullptr;
    if (cudaMalloc(&stage, n * TP_WIRE_G1_BYTES) != cudaSuccess) {
      cudaGetLastError();
      rc = fail(ctx, TP_ERR_CUDA, "srs_deserialize: out of device memory");
    }
    if (rc == TP_OK && cudaMemcpyAsync(stage, bytes + 8, n * TP_WIRE_G1_BYTES, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
      rc = fail(ctx, TP_ERR_CUDA, "srs_deserialize: copy failed");
    if (rc == TP_OK) rc = g1_from_wire_dev(ctx, stage, n, check, s->g1, &rejected, &first);
    if (stage) cudaFree(stage);
    if (rc == TP_OK && rejected) {
      ctx->err = "srs_deserialize: " + std::to_string(rejected) + " G1 point(s) rejected, first at index " + std::to_string(first);
      rc = TP_ERR_MALFORMED;
    }
  }
  if (rc == TP_OK) rc = srs_build_levels_dev(ctx, s);
  if (rc == TP_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, TP_ERR_CUDA, "srs_deserialize: failed");
  if (rc == TP_OK) {
    uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
    g2_encode(q, g2);
    g2_encode(qs, g2s);
    if (tp_srs_set_g2(s, g2, g2s) != TP_OK) rc = fail(ctx, TP_ERR_MALFORMED, "srs_deserialize: G2 points rejected");
  }
  if (rc != TP_OK) {
    tp_srs_destroy(ctx, s);
    return rc;
  }
  *out = s;
  return TP_OK;
}

}  // extern "C"
