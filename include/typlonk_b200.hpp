// typlonk_b200.hpp -- C++17 host side above the C ABI (typlonk_b200.h), header only.
//
// The reference is compiled Rust with no FFI of its own; where its toolchain is absent this is the host language
// that stands in for the Rust shim of INTEGRATION.md.  It mirrors the public API of the three crates name for name
// so that a program written against fabrizio-m/TyPLONK reads the same here:
//
//   kzg          Srs::{from_secret, random, g1_ref, g2_ref, g2s_ref}            kzg/src/srs.rs:8-52
//                (additive: Srs::{contribute, verify, verify_update}, a powers-of-tau ceremony)
//                KzgScheme::{commit, open, verify, identity}                    kzg/src/lib.rs:33-86
//   permutation  Tag, PermutationBuilder::{with_rows, add_row, add_constrain,
//                add_constrains, build}, Permutation::compile,
//                CompiledPermutation::prove                                     permutation/src/lib.rs:12-195, proving.rs:7-31
//   plonk        CircuitDescription (run / build), Var (+, *, clone, assert_eq),
//                CompiledCircuit::{prove, verify, rows}, Proof                  plonk/src/description.rs:4-16, lib.rs:18-35,
//                                                                               proof.rs:26-63, 85-95
//
//   struct Pythagoras {                                   // README.md:16-27
//     static constexpr size_t INPUTS = 3;
//     template <class V> static void run(std::array<V, 3> in) {
//       auto [a, b, c] = in;
//       a = a.clone() * a;  b = b.clone() * b;  c = c.clone() * c;
//       auto d = a + b;
//       d.assert_eq(c);
//     }
//   };
//   typlonk::Context ctx;                                  // one CUDA device; there is no CPU fallback
//   auto circuit = typlonk::build<Pythagoras>(ctx);        // Circuit::build()
//   auto proof = circuit.prove({3, 4, 5}, {0});            // circuit.prove([3, 4, 5], vec![0])
//   assert(circuit.verify(proof));
//
// Where the reference panics, this throws typlonk::Error (code = the C ABI status).  Where the reference draws from
// thread_rng (tau in Srs::random, the nine blinders in prove) there is an overload that takes the values explicitly
// -- the parity tests need them fixed -- and one that draws them from the operating system's CSPRNG (getrandom).
#pragma once

#include <array>
#include <cstdint>
#include <cstring>
#include <memory>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#if defined(__linux__)
#include <sys/random.h>
#endif

#include "typlonk_b200.h"

namespace typlonk {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& what) : std::runtime_error(what + " (status " + std::to_string(c) + ")"), code(c) {}
};
/// `vanishes` assert of plonk/src/proof.rs:321 (TP_ERR_GATE_UNSATISFIED).
struct GateUnsatisfied : Error {
  using Error::Error;
};
/// A wire encoding that is not canonical / not on the curve (TP_ERR_MALFORMED).
struct Malformed : Error {
  using Error::Error;
};

namespace detail {
inline void check(int rc, const char* what, tp_ctx* ctx = nullptr) {
  if (rc == TP_OK) return;
  std::string msg = what;
  if (ctx) {
    const char* e = tp_last_error(ctx);
    if (e && *e) msg += std::string(": ") + e;
  }
  if (rc == TP_ERR_GATE_UNSATISFIED) throw GateUnsatisfied(rc, msg);
  if (rc == TP_ERR_MALFORMED) throw Malformed(rc, msg);
  throw Error(rc, msg);
}
/// 64 bits from the operating system's CSPRNG: getrandom(2) where it exists, else /dev/urandom.
inline uint64_t os_random_u64() {
  uint64_t v = 0;
  size_t got = 0;
#if defined(__linux__)
  while (got < sizeof(v)) {
    ssize_t k = getrandom(reinterpret_cast<unsigned char*>(&v) + got, sizeof(v) - got, 0);
    if (k <= 0) break;
    got += (size_t)k;
  }
#endif
  if (got < sizeof(v)) {
    std::FILE* f = std::fopen("/dev/urandom", "rb");
    if (f) {
      got += std::fread(reinterpret_cast<unsigned char*>(&v) + got, 1, sizeof(v) - got, f);
      std::fclose(f);
    }
  }
  if (got < sizeof(v)) throw Error(TP_ERR_INVALID_ARG, "no operating-system entropy source (getrandom, /dev/urandom)");
  return v;
}
}  // namespace detail

/// BLS12-381 scalar field element: four little-endian u64 limbs in Montgomery form, the memory layout of
/// ark_ff::Fp256 -- buffers of Fr cross the C ABI without conversion.
struct Fr {
  uint64_t limbs[4] = {0, 0, 0, 0};

  Fr() = default;
  /// `Fr::from(i64)`; negative values are r - |v| (plonk/src/utils.rs:152-153).
  Fr(long long v) { detail::check(tp_fr_from_i64((int64_t)v, limbs), "tp_fr_from_i64"); }  // NOLINT(google-explicit-constructor)
  Fr(int v) : Fr((long long)v) {}                                                          // NOLINT(google-explicit-constructor)
  static Fr zero() { return Fr(); }
  static Fr from_canonical(const std::array<uint8_t, 32>& le) {
    Fr r;
    detail::check(tp_fr_from_canonical(le.data(), r.limbs), "tp_fr_from_canonical");
    return r;
  }
  std::array<uint8_t, 32> to_canonical() const {
    std::array<uint8_t, 32> out{};
    detail::check(tp_fr_to_canonical(limbs, out.data()), "tp_fr_to_canonical");
    return out;
  }
  /// ark-ff 0.3 `Fr::rand`: draw 4 x u64, clear the top bit, accept when below r; the accepted limbs ARE the
  /// Montgomery representation (SURVEY.md App. A.4).  `next_u64` is any callable returning uint64_t.
  template <class NextU64>
  static Fr rand(NextU64&& next_u64) {
    static const uint64_t r[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
    for (;;) {
      Fr x;
      for (auto& l : x.limbs) l = next_u64();
      x.limbs[3] &= ~(1ull << 63);
      for (int i = 3; i >= 0; i--) {
        if (x.limbs[i] < r[i]) return x;
        if (x.limbs[i] > r[i]) break;
      }
    }
  }
  /// `Fr::rand(&mut thread_rng())`: every 64-bit word comes straight from the operating system's CSPRNG
  /// (getrandom(2), /dev/urandom as the fallback) -- tau and the blinders are secrets, so no seeded
  /// non-cryptographic generator sits in between.  Throws if the system has no entropy source.
  static Fr random() {
    return rand([] { return detail::os_random_u64(); });
  }
  /// `count` draws of `StdRng::seed_from_u64(seed)` (the generator of plonk/src/proof/challenges.rs:38-45).
  static std::vector<Fr> rand_stream(uint64_t seed, size_t count) {
    std::vector<Fr> out(count);
    if (count) detail::check(tp_fr_rand_stream(seed, count, out[0].limbs), "tp_fr_rand_stream");
    return out;
  }
  bool operator==(const Fr& o) const { return std::memcmp(limbs, o.limbs, 32) == 0; }
  bool operator!=(const Fr& o) const { return !(*this == o); }
};
static_assert(sizeof(Fr) == 32, "Fr must be four packed u64 limbs");

/// Dense polynomial, coefficient form, lowest degree first (ark_poly DensePolynomial<Fr>).
using Poly = std::vector<Fr>;

/// ark_ec GroupAffine {x, y, infinity} as the ABI carries it: x | y (48 B Montgomery each) | infinity flag.
struct G1Affine {
  std::array<uint8_t, TP_G1_BYTES> bytes{};
  bool is_zero() const { return bytes[96] != 0; }
  bool operator==(const G1Affine& o) const { return bytes == o.bytes; }
  bool operator!=(const G1Affine& o) const { return !(*this == o); }
};
struct G2Affine {
  std::array<uint8_t, TP_G2_BYTES> bytes{};
  bool operator==(const G2Affine& o) const { return bytes == o.bytes; }
};

/// One CUDA device + stream.  tp_ctx_create fails with TP_ERR_NO_DEVICE when there is none: no CPU fallback.
class Context {
 public:
  explicit Context(int device = 0, void* cuda_stream = nullptr) {
    tp_ctx* h = nullptr;
    detail::check(tp_ctx_create(device, cuda_stream, &h), "tp_ctx_create (no CUDA device? there is no CPU fallback)");
    h_ = std::shared_ptr<tp_ctx>(h, [](tp_ctx* p) { tp_ctx_destroy(p); });
  }
  /// One context over several GPUs of this process (tp_ctx_create_multi): CompiledCircuit::prove stays ONE call
  /// (plonk/src/proof.rs:26-57) while every MSM, the quotient and the witness upload are sharded over the devices.
  /// A device listed twice = two ranks on it (peer copies instead of NCCL; for tests on one GPU).
  static Context multi(const std::vector<int>& devices) {
    tp_ctx* h = nullptr;
    detail::check(tp_ctx_create_multi(devices.data(), (int)devices.size(), &h), "tp_ctx_create_multi");
    Context c{std::shared_ptr<tp_ctx>(h, [](tp_ctx* p) { tp_ctx_destroy(p); })};
    return c;
  }
  /// ranks behind this context (1 for a single device)
  int ranks() const {
    int n = 1;
    tp_ctx_group_size(get(), &n, nullptr);
    return n;
  }
  tp_ctx* get() const { return h_.get(); }
  void sync() const { detail::check(tp_sync(get()), "tp_sync", get()); }
  uint64_t launch_count() const {
    uint64_t v = 0;
    tp_launch_count(get(), &v);
    return v;
  }

 private:
  explicit Context(std::shared_ptr<tp_ctx> h) : h_(std::move(h)) {}
  std::shared_ptr<tp_ctx> h_;
};

// ---- kzg crate -------------------------------------------------------------------------------------------------------

/// kzg/src/srs.rs:8-52.  The G1 powers live on the device (with the MSM's fixed-base tables).
class Srs {
 public:
  /// Srs::from_secret (srs.rs:30-34): gates + 3 powers, generated on the device.
  static Srs from_secret(const Context& ctx, const Fr& s, size_t gates) {
    tp_srs* h = nullptr;
    detail::check(tp_srs_from_secret(ctx.get(), s.limbs, gates, &h), "tp_srs_from_secret", ctx.get());
    return Srs(ctx, h);
  }
  /// Srs::random (srs.rs:36-41).
  static Srs random(const Context& ctx, size_t gates) { return from_secret(ctx, Fr::random(), gates); }
  /// Additive API (SURVEY.md 8 f4): ark-serialize 0.3 uncompressed Vec<G1> | G2 | tau G2, or with compressed points
  /// (48 B per G1, 96 B per G2; decompressed and checked on the device).
  static Srs from_bytes(const Context& ctx, const std::vector<uint8_t>& raw, int check = 2, bool compressed = false) {
    tp_srs* h = nullptr;
    if (compressed)
      detail::check(tp_srs_deserialize_compressed(ctx.get(), raw.data(), raw.size(), check, &h),
                    "tp_srs_deserialize_compressed", ctx.get());
    else
      detail::check(tp_srs_deserialize(ctx.get(), raw.data(), raw.size(), check, &h), "tp_srs_deserialize", ctx.get());
    return Srs(ctx, h);
  }
  std::vector<uint8_t> to_bytes(bool compressed = false) const {
    size_t need = 0;
    if (compressed) {
      detail::check(tp_srs_serialized_size_compressed(get(), &need), "tp_srs_serialized_size_compressed");
      std::vector<uint8_t> out(need);
      detail::check(tp_srs_serialize_compressed(ctx_.get(), get(), out.data(), out.size(), nullptr),
                    "tp_srs_serialize_compressed", ctx_.get());
      return out;
    }
    detail::check(tp_srs_serialized_size(get(), &need), "tp_srs_serialized_size");
    std::vector<uint8_t> out(need);
    detail::check(tp_srs_serialize(ctx_.get(), get(), out.data(), out.size(), nullptr), "tp_srs_serialize", ctx_.get());
    return out;
  }
  size_t len() const {
    size_t n = 0;
    tp_srs_len(get(), &n);
    return n;
  }
  /// g1_ref (srs.rs:43-45): `count` points from `offset`, as ABI records.
  std::vector<G1Affine> g1_ref(size_t offset = 0, size_t count = SIZE_MAX) const {
    if (count == SIZE_MAX) count = len() - offset;
    std::vector<uint8_t> raw(count * 96);
    detail::check(tp_srs_g1_download(ctx_.get(), get(), offset, count, raw.data()), "tp_srs_g1_download", ctx_.get());
    std::vector<G1Affine> out(count);
    for (size_t i = 0; i < count; i++) {
      bool inf = true;
      for (size_t b = 0; b < 96 && inf; b++) inf = raw[i * 96 + b] == 0;
      if (inf) {  // the device keeps infinity as the all-zero record; GroupAffine::zero() is (0, 1, infinity = true)
        static const uint64_t fq_one[6] = {0x760900000002fffdull, 0xebf4000bc40c0002ull, 0x5f48985753c758baull,
                                           0x77ce585370525745ull, 0x5c071a97a256ec6dull, 0x15f65ec3fa80e493ull};  // R mod q
        std::memcpy(out[i].bytes.data() + 48, fq_one, 48);
        out[i].bytes[96] = 1;
      } else {
        std::memcpy(out[i].bytes.data(), &raw[i * 96], 96);
      }
    }
    return out;
  }
  G2Affine g2_ref() const { return g2_pair().first; }    // srs.rs:46-48
  G2Affine g2s_ref() const { return g2_pair().second; }  // srs.rs:49-51
  /// Additive API, one powers-of-tau contribution (tp_srs_contribute): a new SRS with g1[i] * s^i and g2s * s, and the
  /// pubkey [s]G2 that links it to this one (verify_update).  This SRS is unchanged.
  std::pair<Srs, G2Affine> contribute(const Fr& s) const {
    tp_srs* h = nullptr;
    G2Affine pub;
    detail::check(tp_srs_contribute(ctx_.get(), get(), s.limbs, &h, pub.bytes.data()), "tp_srs_contribute", ctx_.get());
    return {Srs(ctx_, h), pub};
  }
  /// ... with s drawn from the operating system's CSPRNG and forgotten.
  std::pair<Srs, G2Affine> contribute() const { return contribute(Fr::random()); }
  /// Is this SRS the powers of one secret (tp_srs_verify: subgroup checks and a randomised pairing check)?
  bool verify() const {
    int ok = 0;
    detail::check(tp_srs_verify(ctx_.get(), get(), &ok), "tp_srs_verify", ctx_.get());
    return ok != 0;
  }
  /// Was this SRS made from `prev` by the contribution with this pubkey (tp_srs_update_check on g1[1] of both)?
  bool verify_update(const Srs& prev, const G2Affine& pubkey) const {
    int ok = 0;
    detail::check(tp_srs_update_check(prev.g1_ref(1, 1)[0].bytes.data(), g1_ref(1, 1)[0].bytes.data(), pubkey.bytes.data(), &ok),
                  "tp_srs_update_check");
    return ok != 0;
  }
  tp_srs* get() const { return h_.get(); }
  const Context& context() const { return ctx_; }

 private:
  Srs(const Context& ctx, tp_srs* h) : ctx_(ctx) {
    Context keep = ctx;
    h_ = std::shared_ptr<tp_srs>(h, [keep](tp_srs* p) { tp_srs_destroy(keep.get(), p); });
  }
  std::pair<G2Affine, G2Affine> g2_pair() const {
    std::pair<G2Affine, G2Affine> p;
    detail::check(tp_srs_g2(get(), p.first.bytes.data(), p.second.bytes.data()), "tp_srs_g2");
    return p;
  }
  Context ctx_;
  std::shared_ptr<tp_srs> h_;
};

struct KzgCommitment {  // kzg/src/lib.rs:14-20
  G1Affine point;
  const G1Affine& inner() const { return point; }
  bool operator==(const KzgCommitment& o) const { return point == o.point; }
};
struct KzgOpening {  // kzg/src/lib.rs:22-31: (witness commitment, evaluation)
  G1Affine w;
  Fr y;
  const Fr& eval() const { return y; }
};

/// kzg/src/lib.rs:33-86.
class KzgScheme {
 public:
  explicit KzgScheme(const Srs& srs) : srs_(srs) {}
  /// commit (lib.rs:37-54): trailing zero coefficients are stripped as DensePolynomial does; a polynomial longer
  /// than the SRS throws where the reference asserts (lib.rs:43).
  KzgCommitment commit(const Poly& p) const {
    size_t len = stripped(p);
    KzgCommitment c;
    tp_ctx* ctx = srs_.context().get();
    detail::check(tp_commit(ctx, srs_.get(), len ? p[0].limbs : nullptr, len, c.point.bytes.data()), "tp_commit", ctx);
    return c;
  }
  /// open (lib.rs:55-64); the empty polynomial throws like `.expect("at least 1")`.
  KzgOpening open(const Poly& p, const Fr& z) const {
    size_t len = stripped(p);
    KzgOpening o;
    tp_ctx* ctx = srs_.context().get();
    detail::check(tp_open(ctx, srs_.get(), len ? p[0].limbs : nullptr, len, z.limbs, o.w.bytes.data(), o.y.limbs), "tp_open", ctx);
    return o;
  }
  /// verify (lib.rs:66-81).
  bool verify(const KzgCommitment& c, const KzgOpening& o, const Fr& z) const {
    int ok = 0;
    detail::check(tp_kzg_verify(srs_.g2_ref().bytes.data(), srs_.g2s_ref().bytes.data(), c.point.bytes.data(), o.w.bytes.data(),
                                o.y.limbs, z.limbs, &ok),
                  "tp_kzg_verify");
    return ok != 0;
  }
  /// identity (lib.rs:82-85) = commit(1).
  KzgCommitment identity() const { return commit(Poly{Fr(1)}); }

 private:
  static size_t stripped(const Poly& p) {
    size_t len = p.size();
    const Fr z;
    while (len && p[len - 1] == z) len--;
    return len;
  }
  Srs srs_;
};

// ---- permutation crate -----------------------------------------------------------------------------------------------

struct Tag {  // permutation/src/lib.rs:12-26
  size_t i, j;
};
class CompiledPermutation;
/// permutation/src/lib.rs:95-99: the flat map, index = j + i * rows.
struct Permutation {
  std::vector<uint64_t> perm;
  size_t rows() const { return perm.size() / 3; }
  inline CompiledPermutation compile(const Context& ctx) const;  // lib.rs:101-128
};
/// permutation/src/lib.rs:28-93 over the library's native builder.
class PermutationBuilder {
 public:
  PermutationBuilder() : PermutationBuilder(0) {}
  static PermutationBuilder with_rows(size_t rows) { return PermutationBuilder(rows); }
  void add_row() { tp_permutation_builder_add_row(h_.get()); }
  /// Result<(), ()>: false for a tag outside the table (lib.rs:44-56).
  bool add_constrain(Tag left, Tag right) {
    int rc = tp_permutation_builder_add_constrain(h_.get(), left.i, left.j, right.i, right.j);
    if (rc == TP_ERR_INVALID_TAG) return false;
    detail::check(rc, "tp_permutation_builder_add_constrain");
    return true;
  }
  /// `.unwrap()`s every add_constrain (lib.rs:57-61).
  void add_constrains(const std::vector<std::pair<Tag, Tag>>& cs) {
    for (auto& c : cs)
      if (!add_constrain(c.first, c.second)) throw Error(TP_ERR_INVALID_TAG, "add_constrains: called `Result::unwrap()` on an `Err` value");
  }
  Permutation build(size_t size) {
    Permutation p;
    p.perm.resize(3 * size);
    detail::check(tp_permutation_builder_build(h_.get(), size, p.perm.data()), "tp_permutation_builder_build");
    return p;
  }

 private:
  explicit PermutationBuilder(size_t rows) {
    tp_permutation_builder* h = nullptr;
    detail::check(tp_permutation_builder_create(rows, &h), "tp_permutation_builder_create");
    h_ = std::shared_ptr<tp_permutation_builder>(h, [](tp_permutation_builder* p) { tp_permutation_builder_destroy(p); });
  }
  std::shared_ptr<tp_permutation_builder> h_;
};
/// permutation/src/lib.rs:156-195: per column the (id, sigma) values over the domain, and the coset representatives.
class CompiledPermutation {
 public:
  std::array<std::vector<Fr>, 3> id, sigma;
  std::array<Fr, 3> cosets;
  size_t rows = 0;
  /// prove (proving.rs:7-31): rows + 1 running products, out[0] = 1; a zero denominator throws where Fr division panics.
  std::vector<Fr> prove(const std::array<std::vector<Fr>, 3>& values, const Fr& beta, const Fr& gamma) const {
    const uint64_t* v[3] = {values[0][0].limbs, values[1][0].limbs, values[2][0].limbs};
    const uint64_t* ip[3] = {id[0][0].limbs, id[1][0].limbs, id[2][0].limbs};
    const uint64_t* sp[3] = {sigma[0][0].limbs, sigma[1][0].limbs, sigma[2][0].limbs};
    std::vector<Fr> out(rows + 1);
    detail::check(tp_perm_prove(ctx_.get(), v, ip, sp, rows, beta.limbs, gamma.limbs, out[0].limbs), "tp_perm_prove", ctx_.get());
    return out;
  }

 private:
  friend struct Permutation;
  explicit CompiledPermutation(const Context& ctx) : ctx_(ctx) {}
  Context ctx_;
};
inline CompiledPermutation Permutation::compile(const Context& ctx) const {
  CompiledPermutation c(ctx);
  c.rows = rows();
  uint64_t* ip[3];
  uint64_t* sp[3];
  for (int i = 0; i < 3; i++) {
    c.id[i].resize(c.rows);
    c.sigma[i].resize(c.rows);
    ip[i] = c.id[i][0].limbs;
    sp[i] = c.sigma[i][0].limbs;
  }
  uint64_t k[3][4];
  detail::check(tp_permutation_compile(ctx.get(), perm.data(), c.rows, ip, sp, k), "tp_permutation_compile", ctx.get());
  for (int i = 0; i < 3; i++) std::memcpy(c.cosets[i].limbs, k[i], 32);
  return c;
}

// ---- plonk crate -----------------------------------------------------------------------------------------------------

/// description.rs:10-16 `Var`: `+`, `*`, `clone`, `assert_eq`.  A variable is an id in the library's native trace
/// (csrc/trace.cpp), which records the closure ONCE; witnesses are replayed from the recording.
class Var {
 public:
  Var clone() const { return *this; }
  friend Var operator+(const Var& a, const Var& b) { return a.binary(TP_GATE_ADD, b); }
  friend Var operator*(const Var& a, const Var& b) { return a.binary(TP_GATE_MUL, b); }
  void assert_eq(const Var& other) const { detail::check(tp_trace_assert_eq(t_.get(), id_, other.id_), "tp_trace_assert_eq"); }
  uint64_t id() const { return id_; }

 private:
  template <class D>
  friend class CompiledCircuit;
  Var(std::shared_ptr<tp_trace> t, uint64_t id) : t_(std::move(t)), id_(id) {}
  Var binary(int kind, const Var& rhs) const {
    uint64_t out = 0;
    detail::check(tp_trace_gate(t_.get(), kind, id_, rhs.id_, &out), "tp_trace_gate");
    return Var(t_, out);
  }
  std::shared_ptr<tp_trace> t_;
  uint64_t id_;
};

/// proof.rs:85-95.  `fixed` is the 1472-byte block of tp_prove (13 G1 + 7 Fr, ark-serialize 0.3 uncompressed).
struct Proof {
  std::array<uint8_t, TP_PROOF_FIXED_BYTES> fixed{};
  std::vector<Fr> public_inputs;  // padded to `rows` (proof.rs:52-53, 190)
  /// Additive API (SURVEY.md 8 f4).  compressed: the same framing with an 848-byte block of compressed points.
  std::vector<uint8_t> to_bytes(bool compressed = false) const {
    size_t need = 0;
    const uint64_t* pis = public_inputs.empty() ? nullptr : public_inputs[0].limbs;
    if (compressed) {
      tp_proof_encoded_size_compressed(public_inputs.size(), &need);
      std::vector<uint8_t> out(need);
      detail::check(tp_proof_encode_compressed(fixed.data(), pis, public_inputs.size(), out.data(), out.size(), nullptr),
                    "tp_proof_encode_compressed");
      return out;
    }
    tp_proof_encoded_size(public_inputs.size(), &need);
    std::vector<uint8_t> out(need);
    detail::check(tp_proof_encode(fixed.data(), pis, public_inputs.size(), out.data(), out.size(), nullptr),
                  "tp_proof_encode");
    return out;
  }
  /// `fixed` is the uncompressed block either way.
  static Proof from_bytes(const std::vector<uint8_t>& raw, bool compressed = false) {
    auto decode = compressed ? tp_proof_decode_compressed : tp_proof_decode;
    const char* what = compressed ? "tp_proof_decode_compressed" : "tp_proof_decode";
    Proof p;
    size_t n = 0;
    detail::check(decode(raw.data(), raw.size(), nullptr, nullptr, 0, &n), what);
    p.public_inputs.resize(n);
    detail::check(decode(raw.data(), raw.size(), p.fixed.data(), n ? p.public_inputs[0].limbs : nullptr, n, &n), what);
    return p;
  }
  /// tp_proofs_decompress: `count` contiguous compressed blocks -> uncompressed blocks, the square roots on the device.
  /// status[k] is TP_OK or TP_ERR_MALFORMED (block zero-filled); without `status` a malformed block throws.
  static std::vector<std::array<uint8_t, TP_PROOF_FIXED_BYTES>> decompress_blocks(const Context& ctx,
                                                                                 const std::vector<uint8_t>& blocks,
                                                                                 std::vector<int>* status = nullptr) {
    const size_t count = blocks.size() / TP_PROOF_COMPRESSED_FIXED_BYTES;
    if (count * TP_PROOF_COMPRESSED_FIXED_BYTES != blocks.size())
      throw Malformed(TP_ERR_MALFORMED, "decompress_blocks: not a whole number of compressed proof blocks");
    std::vector<std::array<uint8_t, TP_PROOF_FIXED_BYTES>> out(count);
    if (status) status->assign(count, TP_OK);
    detail::check(tp_proofs_decompress(ctx.get(), blocks.data(), count, count ? out[0].data() : nullptr,
                                       count * TP_PROOF_FIXED_BYTES, status ? status->data() : nullptr),
                  "tp_proofs_decompress", ctx.get());
    return out;
  }
};

/// Additive API: what verify() reads of a compiled circuit (tp_vk_*): n, the cosets, the eight commitments, srs[0], the
/// SRS's G2 points and sigma_1, sigma_2 in coefficient form, so 1376 + 64n bytes on the wire.
class VerifyingKey {
 public:
  /// tp_vk_deserialize; check 0 / 1 / 2 as Srs::from_bytes.  A rejected key throws Malformed naming the field.
  static VerifyingKey from_bytes(const Context& ctx, const std::vector<uint8_t>& raw, int check = 2) {
    tp_vk* h = nullptr;
    detail::check(tp_vk_deserialize(ctx.get(), raw.data(), raw.size(), check, &h), "tp_vk_deserialize", ctx.get());
    return VerifyingKey(ctx, h);
  }
  std::vector<uint8_t> to_bytes() const {
    size_t need = 0;
    tp_vk_serialized_size(get(), &need);
    std::vector<uint8_t> out(need);
    detail::check(tp_vk_serialize(ctx_.get(), get(), out.data(), out.size(), nullptr), "tp_vk_serialize", ctx_.get());
    return out;
  }
  /// CompiledCircuit::verify against the key (tp_vk_verify): the same verdict, and the same throws.
  bool verify(const Proof& proof) const {
    int ok = 0;
    detail::check(tp_vk_verify(ctx_.get(), get(), proof.fixed.data(), proof.fixed.size(),
                               proof.public_inputs.empty() ? nullptr : proof.public_inputs[0].limbs, proof.public_inputs.size(), &ok),
                  "tp_vk_verify", ctx_.get());
    return ok != 0;
  }
  tp_vk* get() const { return h_.get(); }
  const Context& context() const { return ctx_; }

 private:
  template <class D>
  friend class CompiledCircuit;
  VerifyingKey(const Context& ctx, tp_vk* h) : ctx_(ctx) {
    Context keep = ctx;
    h_ = std::shared_ptr<tp_vk>(h, [keep](tp_vk* p) { tp_vk_destroy(keep.get(), p); });
  }
  Context ctx_;
  std::shared_ptr<tp_vk> h_;
};

/// Additive API: proofs of several circuits in one folded check (tp_vk_verify_batch) -> per-proof verdicts.  The keys
/// must share one context; they may differ in size and SRS.
inline std::vector<bool> verify_batch(const std::vector<std::pair<const VerifyingKey*, const Proof*>>& pairs) {
  if (pairs.empty()) return {};
  std::vector<tp_vk*> keys;
  std::vector<uint32_t> key_of(pairs.size());
  std::vector<uint8_t> blob(pairs.size() * TP_PROOF_FIXED_BYTES);
  std::vector<const uint64_t*> pis(pairs.size());
  std::vector<size_t> npub(pairs.size());
  for (size_t k = 0; k < pairs.size(); k++) {
    tp_vk* h = pairs[k].first->get();
    size_t j = 0;
    while (j < keys.size() && keys[j] != h) j++;
    if (j == keys.size()) keys.push_back(h);
    key_of[k] = (uint32_t)j;
    const Proof& p = *pairs[k].second;
    std::memcpy(blob.data() + k * TP_PROOF_FIXED_BYTES, p.fixed.data(), TP_PROOF_FIXED_BYTES);
    pis[k] = p.public_inputs.empty() ? nullptr : p.public_inputs[0].limbs;
    npub[k] = p.public_inputs.size();
  }
  tp_ctx* ctx = pairs[0].first->context().get();
  int all_ok = 0;
  std::vector<int> each(pairs.size());
  detail::check(tp_vk_verify_batch(ctx, keys.data(), keys.size(), key_of.data(), blob.data(), pairs.size(), pis.data(),
                                   npub.data(), &all_ok, each.data()),
                "tp_vk_verify_batch", ctx);
  return std::vector<bool>(each.begin(), each.end());
}

/// plonk/src/lib.rs:18-35.  DESC provides `static constexpr size_t INPUTS` and
/// `template <class V> static void run(std::array<V, INPUTS>)` (description.rs:4-9).
template <class DESC>
class CompiledCircuit {
 public:
  static constexpr size_t INPUTS = DESC::INPUTS;
  size_t rows = 0;
  std::array<KzgCommitment, 5> fixed_commitments;

  /// CircuitBuilder::compile (builder.rs:60-113) with the SRS secret as an input.
  CompiledCircuit(const Context& ctx, const Fr& tau) : ctx_(ctx) {
    trace();
    compile(Srs::from_secret(ctx, tau, rows));
  }
  /// Additive API: compiled against an existing SRS (e.g. the outcome of a ceremony) of at least `rows` points.
  CompiledCircuit(const Context& ctx, const Srs& srs) : ctx_(ctx) {
    trace();
    compile(srs);
  }

  /// CompiledCircuit::prove (proof.rs:26-57) with the nine blinders a0 a1 a2 b0 b1 b2 c0 c1 c2 (proof.rs:43-48)
  /// given.  Throws GateUnsatisfied where the reference panics in `vanishes`.
  Proof prove(const std::array<Fr, INPUTS>& inputs, const std::vector<Fr>& public_inputs, const std::array<Fr, 9>& blinders) const {
    if (public_inputs.size() > rows) throw Error(TP_ERR_INVALID_ARG, "prove: more public inputs than rows");
    std::vector<Fr> a(rows), b(rows), c(rows);
    uint64_t* adv[3] = {a[0].limbs, b[0].limbs, c[0].limbs};
    detail::check(tp_trace_witness(trace_.get(), INPUTS ? inputs[0].limbs : nullptr, INPUTS, blinders[0].limbs, adv), "tp_trace_witness");
    Proof p;
    const uint64_t* cadv[3] = {adv[0], adv[1], adv[2]};
    detail::check(tp_prove_inputs(ctx_.get(), circuit_.get(), cadv, public_inputs.empty() ? nullptr : public_inputs[0].limbs,
                                  public_inputs.size(), p.fixed.data(), p.fixed.size()),
                  "tp_prove", ctx_.get());
    p.public_inputs = public_inputs;
    p.public_inputs.resize(rows);
    return p;
  }
  /// ... with the blinders drawn like `Fr::rand(&mut thread_rng())`.
  Proof prove(const std::array<Fr, INPUTS>& inputs, const std::vector<Fr>& public_inputs) const {
    std::array<Fr, 9> blinders;
    for (auto& x : blinders) x = Fr::random();
    return prove(inputs, public_inputs, blinders);
  }
  /// Many proofs in one call (tp_prove_batch): proof k equals prove(inputs[k], public_inputs[k], blinders[k]).  Throws
  /// what prove() would throw for the first failing proof; tp_last_error names its index.
  std::vector<Proof> prove_batch(const std::vector<std::array<Fr, INPUTS>>& inputs, const std::vector<std::vector<Fr>>& public_inputs,
                                 const std::vector<std::array<Fr, 9>>& blinders) const {
    const size_t count = inputs.size();
    if (public_inputs.size() != count || blinders.size() != count)
      throw Error(TP_ERR_INVALID_ARG, "prove_batch: inputs, public inputs and blinders differ in count");
    std::vector<Fr> cols(3 * count * rows);
    std::vector<const uint64_t*> adv(3 * count);
    std::vector<const uint64_t*> pis(count);
    std::vector<size_t> npub(count);
    for (size_t k = 0; k < count; k++) {
      if (public_inputs[k].size() > rows) throw Error(TP_ERR_INVALID_ARG, "prove_batch: more public inputs than rows");
      uint64_t* a[3];
      for (int i = 0; i < 3; i++) adv[3 * k + i] = a[i] = cols[(3 * k + i) * rows].limbs;
      detail::check(tp_trace_witness(trace_.get(), INPUTS ? inputs[k][0].limbs : nullptr, INPUTS, blinders[k][0].limbs, a), "tp_trace_witness");
      pis[k] = public_inputs[k].empty() ? nullptr : public_inputs[k][0].limbs;
      npub[k] = public_inputs[k].size();
    }
    std::vector<uint8_t> blob(count * TP_PROOF_FIXED_BYTES);
    detail::check(tp_prove_batch(ctx_.get(), circuit_.get(), count, adv.data(), pis.data(), npub.data(), blob.data(), blob.size(), nullptr),
                  "tp_prove_batch", ctx_.get());
    std::vector<Proof> out(count);
    for (size_t k = 0; k < count; k++) {
      std::memcpy(out[k].fixed.data(), blob.data() + k * TP_PROOF_FIXED_BYTES, TP_PROOF_FIXED_BYTES);
      out[k].public_inputs = public_inputs[k];
      out[k].public_inputs.resize(rows);
    }
    return out;
  }
  /// CompiledCircuit::verify (proof.rs:59-63, 195-233).  A malformed proof throws; a wrong one returns false.
  bool verify(const Proof& proof) const {
    int ok = 0;
    detail::check(tp_verify(ctx_.get(), circuit_.get(), proof.fixed.data(), proof.fixed.size(),
                            proof.public_inputs.empty() ? nullptr : proof.public_inputs[0].limbs, proof.public_inputs.size(), &ok),
                  "tp_verify", ctx_.get());
    return ok != 0;
  }
  /// Additive API: every proof checked at once (tp_verify_batch) -> per-proof verdicts.  Stricter than verify() on
  /// points outside the prime-order subgroup, which it rejects.
  std::vector<bool> verify_batch(const std::vector<Proof>& proofs) const {
    std::vector<uint8_t> blob(proofs.size() * TP_PROOF_FIXED_BYTES);
    std::vector<const uint64_t*> pis(proofs.size());
    std::vector<size_t> npub(proofs.size());
    for (size_t k = 0; k < proofs.size(); k++) {
      std::memcpy(blob.data() + k * TP_PROOF_FIXED_BYTES, proofs[k].fixed.data(), TP_PROOF_FIXED_BYTES);
      pis[k] = proofs[k].public_inputs.empty() ? nullptr : proofs[k].public_inputs[0].limbs;
      npub[k] = proofs[k].public_inputs.size();
    }
    int all_ok = 0;
    std::vector<int> each(proofs.size());
    detail::check(tp_verify_batch(ctx_.get(), circuit_.get(), blob.data(), proofs.size(), pis.data(), npub.data(), &all_ok,
                                  each.data()),
                  "tp_verify_batch", ctx_.get());
    return std::vector<bool>(each.begin(), each.end());
  }
  /// Additive API: the circuit's verification key (tp_vk_from_circuit); it outlives the circuit.
  VerifyingKey verifying_key() const {
    tp_vk* h = nullptr;
    detail::check(tp_vk_from_circuit(ctx_.get(), circuit_.get(), &h), "tp_vk_from_circuit", ctx_.get());
    return VerifyingKey(ctx_, h);
  }
  const Srs& srs() const { return *srs_; }
  tp_circuit* get() const { return circuit_.get(); }

 private:
  template <size_t... K>
  std::array<Var, INPUTS> make_inputs(std::index_sequence<K...>) const {
    return {Var(trace_, (uint64_t)K)...};
  }
  void trace() {
    tp_trace* t = nullptr;
    detail::check(tp_trace_create(INPUTS, &t), "tp_trace_create");
    trace_ = std::shared_ptr<tp_trace>(t, [](tp_trace* p) { tp_trace_destroy(p); });
    DESC::template run<Var>(make_inputs(std::make_index_sequence<INPUTS>{}));
    size_t gates = 0;
    detail::check(tp_trace_finish(t, &rows, &gates), "tp_trace_finish (an asserted variable never entered a gate?)");
  }
  void compile(const Srs& srs) {
    srs_ = std::make_unique<Srs>(srs);
    std::vector<Fr> sel(5 * rows);
    detail::check(tp_trace_selectors(trace_.get(), sel[0].limbs), "tp_trace_selectors");
    std::vector<uint64_t> perm(3 * rows);
    detail::check(tp_trace_permutation(trace_.get(), perm.data()), "tp_trace_permutation");
    const uint64_t* cols[5];
    for (int k = 0; k < 5; k++) cols[k] = sel[k * rows].limbs;
    uint8_t fixed[5 * TP_G1_BYTES];
    tp_circuit* c = nullptr;
    detail::check(tp_circuit_compile(ctx_.get(), srs_->get(), cols, perm.data(), rows, &c, fixed), "tp_circuit_compile", ctx_.get());
    Context keep = ctx_;
    circuit_ = std::shared_ptr<tp_circuit>(c, [keep](tp_circuit* p) { tp_circuit_destroy(keep.get(), p); });
    for (int k = 0; k < 5; k++) std::memcpy(fixed_commitments[k].point.bytes.data(), fixed + k * TP_G1_BYTES, TP_G1_BYTES);
  }
  Context ctx_;
  std::shared_ptr<tp_trace> trace_;
  std::unique_ptr<Srs> srs_;
  std::shared_ptr<tp_circuit> circuit_;
};

/// `Circuit::build()` (description.rs:6-8): tau from the thread's random generator like Srs::random (builder.rs:71) ...
template <class DESC>
CompiledCircuit<DESC> build(const Context& ctx) {
  return CompiledCircuit<DESC>(ctx, Fr::random());
}
/// ... or given, for reproducible setups.
template <class DESC>
CompiledCircuit<DESC> build(const Context& ctx, const Fr& tau) {
  return CompiledCircuit<DESC>(ctx, tau);
}
/// ... or on an SRS the caller made, e.g. by a ceremony (Srs::contribute, Srs::verify).
template <class DESC>
CompiledCircuit<DESC> build(const Context& ctx, const Srs& srs) {
  return CompiledCircuit<DESC>(ctx, srs);
}

}  // namespace typlonk
