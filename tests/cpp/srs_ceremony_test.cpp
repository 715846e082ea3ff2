// The SRS ceremony through include/typlonk_b200.hpp: Srs::random -> two contributions -> verify -> verify_update ->
// the README circuit compiled on the result -> prove -> verify.
#include <cstdio>

#include "typlonk_b200.hpp"

using namespace typlonk;

static int failures = 0;
#define CHECK(name, cond)                          \
  do {                                             \
    bool ok__ = (cond);                            \
    std::printf("%s %s\n", ok__ ? "ok  " : "FAIL", name); \
    if (!ok__) failures++;                         \
  } while (0)

struct Pythagoras {  // README.md:16-27
  static constexpr size_t INPUTS = 3;
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
  Context ctx;
  auto start = Srs::random(ctx, 64);
  CHECK("a random SRS verifies", start.verify());
  auto [mid, pk1] = start.contribute();
  auto [last, pk2] = mid.contribute(Fr::rand_stream(5, 1)[0]);
  CHECK("contributed SRSs verify", mid.verify() && last.verify());
  CHECK("each link checks", mid.verify_update(start, pk1) && last.verify_update(mid, pk2));
  CHECK("a link with the wrong pubkey fails", !last.verify_update(mid, pk1) && !mid.verify_update(start, pk2));
  CHECK("the contribution changed the powers", last.g1_ref(1, 1)[0] != start.g1_ref(1, 1)[0] && last.g1_ref(0, 1)[0] == start.g1_ref(0, 1)[0]);
  bool threw = false;
  try {
    start.contribute(Fr::zero());
  } catch (const Error& e) {
    threw = e.code == TP_ERR_INVALID_ARG;
  }
  CHECK("a zero secret throws", threw);

  auto circuit = build<Pythagoras>(ctx, last);
  auto proof = circuit.prove({Fr(3), Fr(4), Fr(5)}, {Fr(0)});
  CHECK("a proof on the ceremony's SRS verifies", circuit.verify(proof));
  bool rejected = true;   // 3^2 + 4^2 != 6^2 breaks a copy constraint: the proof is made, and verify refuses it
  try {
    rejected = !circuit.verify(circuit.prove({Fr(3), Fr(4), Fr(6)}, {Fr(0)}));
  } catch (const GateUnsatisfied&) {
  }
  CHECK("a wrong witness gives no accepted proof", rejected);
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
