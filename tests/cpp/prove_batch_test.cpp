// CompiledCircuit::prove_batch through include/typlonk_b200.hpp: every proof equals prove() on the same inputs, the
// proofs verify, and a witness that breaks the gates throws as prove() does.
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
  std::vector<std::array<Fr, 2>> inputs;
  std::vector<std::vector<Fr>> pis;
  std::vector<std::array<Fr, 9>> blinders;
  for (int k = 0; k < 6; k++) {
    auto b = Fr::rand_stream(100 + k, 9);
    std::array<Fr, 9> bl;
    for (int i = 0; i < 9; i++) bl[i] = b[i];
    inputs.push_back({Fr(3 + k), Fr(5)});
    pis.push_back({Fr(0)});
    blinders.push_back(bl);
  }
  auto batch = circuit.prove_batch(inputs, pis, blinders);
  bool same = batch.size() == inputs.size();
  for (size_t k = 0; same && k < inputs.size(); k++) {
    auto single = circuit.prove(inputs[k], pis[k], blinders[k]);
    same = single.fixed == batch[k].fixed && single.public_inputs == batch[k].public_inputs;
  }
  CHECK("every batch proof equals prove() on the same inputs", same);
  bool all_verify = true;
  for (auto& p : batch) all_verify = all_verify && circuit.verify(p);
  CHECK("batch proofs verify", all_verify);
  pis[4] = {Fr(1)};   // an uncompensated public input: the gate line no longer vanishes
  bool threw = false;
  try {
    circuit.prove_batch(inputs, pis, blinders);
  } catch (const Error& e) {
    threw = e.code == TP_ERR_GATE_UNSATISFIED && std::string(e.what()).find("proof 4") != std::string::npos;
  }
  CHECK("a bad witness throws, naming its index", threw);
  CHECK("empty batch", circuit.prove_batch({}, {}, {}).empty());
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
