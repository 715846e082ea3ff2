// CompiledCircuit::verify_batch through include/typlonk_b200.hpp: a batch of honest proofs is accepted proof by proof,
// a tampered proof is the only one rejected, and the verdicts equal verify()'s.
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

struct MulChain {
  static constexpr size_t INPUTS = 2;
  template <class V>
  static void run(std::array<V, 2> in) {
    auto [x, y] = in;
    for (int i = 0; i < 29; i++) x = x * y.clone();
  }
};

int main() {
  Context ctx;
  const Fr tau = Fr::rand_stream(1, 1)[0];
  auto circuit = build<MulChain>(ctx, tau);
  std::vector<Proof> proofs;
  for (int k = 0; k < 6; k++) {
    auto b = Fr::rand_stream(100 + k, 9);
    std::array<Fr, 9> blinders;
    for (int i = 0; i < 9; i++) blinders[i] = b[i];
    proofs.push_back(circuit.prove({Fr(3 + k), Fr(5)}, {Fr(0)}, blinders));
  }
  auto ok = circuit.verify_batch(proofs);
  CHECK("honest batch: every proof accepted", ok.size() == proofs.size() && ok == std::vector<bool>(proofs.size(), true));
  proofs[4].fixed[192] ^= 1;  // a(zeta)
  ok = circuit.verify_batch(proofs);
  bool same = ok.size() == proofs.size();
  for (size_t k = 0; same && k < proofs.size(); k++) same = ok[k] == (k != 4) && ok[k] == circuit.verify(proofs[k]);
  CHECK("tampered proof 4 alone rejected, as verify() rejects it", same);
  CHECK("empty batch", circuit.verify_batch({}).empty());
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
