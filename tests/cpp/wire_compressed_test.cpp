// Compressed wire encodings through include/typlonk_b200.hpp: the SRS and proofs round-trip through the compressed
// forms, the blocks are the advertised sizes, batch decompression equals the host decoder, and bad bytes throw.
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
  auto srs = Srs::from_secret(ctx, tau, 61);
  auto raw = srs.to_bytes(true);
  CHECK("compressed SRS size", raw.size() == 8 + 64 * TP_WIRE_G1_COMPRESSED_BYTES + 2 * TP_WIRE_G2_COMPRESSED_BYTES);
  auto back = Srs::from_bytes(ctx, raw, 2, true);
  CHECK("compressed SRS round trip", back.to_bytes() == srs.to_bytes() && back.to_bytes(true) == raw);
  auto bad = raw;
  bad[8 + 48 * 3 + 47] |= 0xc0;
  bool threw = false;
  try {
    Srs::from_bytes(ctx, bad, 2, true);
  } catch (const Malformed& e) {
    threw = std::string(e.what()).find("first at index 3") != std::string::npos;
  }
  CHECK("a bad record throws Malformed, naming its index", threw);

  auto circuit = build<MulChain>(ctx, tau);
  auto blinders = Fr::rand_stream(2, 9);
  std::array<Fr, 9> bl;
  for (int i = 0; i < 9; i++) bl[i] = blinders[i];
  auto proof = circuit.prove({Fr(3), Fr(5)}, {Fr(0)}, bl);
  auto enc = proof.to_bytes(true);
  CHECK("compressed proof size", enc.size() == TP_PROOF_COMPRESSED_FIXED_BYTES + 8 + 32 * proof.public_inputs.size());
  auto dec = Proof::from_bytes(enc, true);
  CHECK("compressed proof round trip", dec.fixed == proof.fixed && dec.public_inputs == proof.public_inputs);
  CHECK("decoded proof verifies", circuit.verify(dec));

  std::vector<uint8_t> blocks(enc.begin(), enc.begin() + TP_PROOF_COMPRESSED_FIXED_BYTES);
  blocks.insert(blocks.end(), enc.begin(), enc.begin() + TP_PROOF_COMPRESSED_FIXED_BYTES);
  blocks[TP_PROOF_COMPRESSED_FIXED_BYTES + 47] |= 0xc0;   // second block: both flags on a.commitment
  std::vector<int> status;
  auto fixed = Proof::decompress_blocks(ctx, blocks, &status);
  CHECK("batch decompression: statuses", status.size() == 2 && status[0] == TP_OK && status[1] == TP_ERR_MALFORMED);
  std::array<uint8_t, TP_PROOF_FIXED_BYTES> zero{};
  CHECK("batch decompression: blocks", fixed[0] == proof.fixed && fixed[1] == zero);
  threw = false;
  try {
    Proof::decompress_blocks(ctx, blocks);
  } catch (const Malformed& e) {
    threw = std::string(e.what()).find("proof 1") != std::string::npos;
  }
  CHECK("batch decompression without statuses throws, naming the block", threw);
  std::printf("%d failures\n", failures);
  return failures ? 1 : 0;
}
