// Proof format v2 through include/typlonk_b200.hpp: a circuit with public inputs is traced, its key made and round
// tripped through bytes, a proof made, encoded and decoded, and verified without a context; a wrong public value, a
// tampered proof and a damaged key are rejected, and a witness that breaks a gate throws.
#include <cstdio>
#include <string>

#include "typlonk_b200.hpp"

using namespace typlonk;

static int failures = 0;
#define CHECK(name, cond)                          \
  do {                                             \
    bool ok__ = (cond);                            \
    std::printf("%s %s\n", ok__ ? "ok  " : "FAIL", name); \
    if (!ok__) failures++;                         \
  } while (0)

struct Pythagoras {  // README.md:16-27, with a and c public
  static constexpr size_t INPUTS = 3;
  static constexpr size_t PUBLIC = 3;
  template <class V>
  static void run(std::array<V, 3> in) {
    auto [a, b, c] = in;
    a = a.clone() * a;
    b = b.clone() * b;
    c = c.clone() * c;
    auto d = a + b;
    d.assert_eq(c);
  }
};

int main() {
  std::vector<uint8_t> key_bytes;
  ProofV2 proof;
  {
    Context ctx;
    const Fr tau = Fr::rand_stream(1, 1)[0];
    auto circuit = build<Pythagoras>(ctx, tau);
    key_bytes = circuit.verifying_key_v2().to_bytes();
    CHECK("key is 1368 bytes", key_bytes.size() == TP_VK2_BYTES);
    auto b = Fr::rand_stream(2, 9);
    std::array<Fr, 9> blinders;
    for (int i = 0; i < 9; i++) blinders[i] = b[i];
    proof = circuit.prove_v2({Fr(3), Fr(4), Fr(5)}, blinders);
    CHECK("proof carries the public values", proof.public_inputs.size() == 3 && proof.public_inputs[2] == Fr(5));
    CHECK("circuit's key verifies", circuit.verifying_key_v2().verify(proof));
    // every gate holds, the copy constraint d = c^2 does not: a proof comes out, and it is rejected
    auto broken = circuit.prove_v2({Fr(3), Fr(4), Fr(6)}, blinders);
    CHECK("a copy violation gives a rejected proof", !circuit.verifying_key_v2().verify(broken));
  }
  // no context from here on
  auto vk = VerifyingKeyV2::from_bytes(key_bytes, 2);
  CHECK("key round trip", vk.to_bytes() == key_bytes);
  auto raw = proof.to_bytes();
  CHECK("encoded size", raw.size() == TP_PROOF_V2_FIXED_BYTES + 8 + 3 * 32);
  auto again = ProofV2::from_bytes(raw);
  CHECK("proof round trip", again.fixed == proof.fixed && again.public_inputs == proof.public_inputs);
  CHECK("verifies without a context", vk.verify(again));
  std::vector<Fr> wrong = {Fr(3), Fr(4), Fr(6)};
  CHECK("wrong public value rejected", !vk.verify(again, &wrong));
  ProofV2 bad = again;
  bad.fixed[TP_PROOF_V2_FIXED_BYTES - 1] ^= 1;
  CHECK("tampered evaluation rejected", !vk.verify(bad));
  bool malformed = false;
  try {
    std::vector<uint8_t> cut(raw.begin(), raw.end() - 1);
    ProofV2::from_bytes(cut);
  } catch (const Malformed&) {
    malformed = true;
  }
  CHECK("truncated proof throws Malformed", malformed);
  malformed = false;
  std::string what;
  try {
    std::vector<uint8_t> k = key_bytes;
    k[0] = 'X';
    VerifyingKeyV2::from_bytes(k);
  } catch (const Malformed& e) {
    malformed = true;
    what = e.what();
  }
  CHECK("damaged key throws Malformed naming the tag", malformed && what.find("tag") != std::string::npos);
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
