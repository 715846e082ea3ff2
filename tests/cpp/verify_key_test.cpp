// Verification keys through include/typlonk_b200.hpp: a key exported from a circuit survives a byte round trip,
// verifies like CompiledCircuit::verify, keeps working after the circuit is gone, and checks proofs of two circuits
// of different sizes in one batch, localising a tampered proof.
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

template <int GATES>
struct MulChain {
  static constexpr size_t INPUTS = 2;
  template <class V>
  static void run(std::array<V, 2> in) {
    auto [x, y] = in;
    for (int i = 0; i < GATES; i++) x = x * y.clone();
  }
};

template <class C>
static std::vector<Proof> proofs_of(const C& circuit, int count, int seed) {
  std::vector<Proof> out;
  for (int k = 0; k < count; k++) {
    auto b = Fr::rand_stream(seed + k, 9);
    std::array<Fr, 9> blinders;
    for (int i = 0; i < 9; i++) blinders[i] = b[i];
    out.push_back(circuit.prove({Fr(3 + k), Fr(5)}, {Fr(0)}, blinders));
  }
  return out;
}

int main() {
  Context ctx;
  const Fr tau = Fr::rand_stream(1, 1)[0];
  std::vector<uint8_t> raw_small;
  std::vector<Proof> small_proofs;
  {
    auto small = build<MulChain<29>>(ctx, tau);
    small_proofs = proofs_of(small, 4, 200);
    auto vk = small.verifying_key();
    raw_small = vk.to_bytes();
    CHECK("key size is 1376 + 64n", raw_small.size() == 1376 + 64 * small.rows);
    bool same = true;
    for (auto& p : small_proofs) same = same && vk.verify(p) && small.verify(p);
    Proof bad = small_proofs[1];
    bad.fixed[192] ^= 1;
    CHECK("key verdicts equal verify()", same && !vk.verify(bad) && !small.verify(bad));
  }
  auto vk_small = VerifyingKey::from_bytes(ctx, raw_small, 2);
  CHECK("round trip after the circuit is gone", vk_small.to_bytes() == raw_small);
  CHECK("deserialised key verifies", vk_small.verify(small_proofs[0]));
  auto big = build<MulChain<1000>>(ctx, tau);
  auto vk_big = big.verifying_key();
  auto big_proofs = proofs_of(big, 4, 300);
  std::vector<std::pair<const VerifyingKey*, const Proof*>> pairs;
  for (int k = 0; k < 4; k++) {
    pairs.push_back({&vk_small, &small_proofs[k]});
    pairs.push_back({&vk_big, &big_proofs[k]});
  }
  auto ok = verify_batch(pairs);
  CHECK("two keys, honest batch", ok == std::vector<bool>(8, true));
  Proof bad = big_proofs[2];
  bad.fixed[1024 + 1] ^= 1;
  pairs[5].second = &bad;
  ok = verify_batch(pairs);
  bool localised = ok.size() == 8;
  for (size_t k = 0; localised && k < 8; k++) localised = ok[k] == (k != 5);
  CHECK("tampered proof 5 alone rejected", localised);
  bool threw = false;
  try {
    std::vector<uint8_t> cut(raw_small.begin(), raw_small.end() - 1);
    VerifyingKey::from_bytes(ctx, cut);
  } catch (const Malformed&) {
    threw = true;
  }
  CHECK("truncated key throws Malformed", threw);
  CHECK("empty batch", verify_batch({}).empty());
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
