// Host-side circuit tracing, copy-constraint compilation and witness generation (SURVEY.md 8 f3).
//
// What it stands in for, in the reference:
//   * the tracing DSL's bookkeeping       Context / BuildVar      plonk/src/builder.rs:119-188, 339-378, 427-433
//   * padding to the domain size          CircuitBuilder::fill    plonk/src/builder.rs:47-58
//   * selector columns                    Gate::to_row + compile  plonk/src/builder.rs:73-84, 316-324
//   * copy-constraint cycles              PermutationBuilder      permutation/src/lib.rs:28-93
//   * witness columns                     ComputeVar + prove()    plonk/src/builder.rs:380-397, plonk/src/proof.rs:33-49
//
// The reference walks the circuit closure twice (once over BuildVar to record gates, once per proof over ComputeVar
// to compute values), takes a Mutex and prints a line per gate, and keeps its constraints in a HashMap whose iteration
// order is random per process.  Here a circuit is recorded ONCE as a flat gate list (struct of arrays); the witness
// is a replay of that list over Fr, and the constraint classes are walked in first-insertion order (the order is an
// input, like tau and the blinders -- DESIGN.md 2).  Everything here is sequential by nature (a gate's operands are
// earlier gates' outputs) and stays on the host; the numeric setup and the prover run on the device.
#include <stdint.h>
#include <string.h>

#include <new>
#include <algorithm>
#include <vector>

#include "../../include/typlonk_b200.h"
#include "host_field.h"

using tph::HFr;

namespace {

constexpr uint64_t kNoTag = ~0ull;
constexpr unsigned kColumns = 3;  // PermutationBuilder<3>, builder.rs:27

// (column i, row j) packed so that a tag is one word; j < 2^60.
inline uint64_t pack_tag(uint64_t i, uint64_t j) { return (j << 2) | i; }
inline uint64_t tag_col(uint64_t t) { return t & 3; }
inline uint64_t tag_row(uint64_t t) { return t >> 2; }

// permutation/src/lib.rs:28-93.  Constraints are (class key, member) pairs kept in arrival order; `build` groups
// them by key with a stable counting pass, which reproduces "for (left, rights) in constrains" with the classes in
// first-insertion order and each class's members in push order.
struct CopyConstraints {
  size_t rows = 0;
  std::vector<uint32_t> slot_of;                   // packed key tag -> class number + 1 (0 = none); tags are dense (4 per row)
  std::vector<uint64_t> keys;                      // class number -> key tag
  std::vector<uint32_t> pair_slot;                 // arrival order
  std::vector<uint64_t> pair_right;

  // check_tag: `i <= C && j < rows` (lib.rs:44-47; the `<=` is the reference's)
  bool check(uint64_t col, uint64_t row) const { return col <= kColumns && row < rows; }

  bool add(uint64_t li, uint64_t lj, uint64_t ri, uint64_t rj) {
    if (!check(li, lj) || !check(ri, rj)) return false;
    uint64_t key = pack_tag(li, lj);
    if (key >= slot_of.size()) slot_of.resize(std::max<size_t>(4 * rows, 2 * slot_of.size()), 0);
    uint32_t slot;
    if (slot_of[key] == 0) {
      slot = (uint32_t)keys.size();
      slot_of[key] = slot + 1;
      keys.push_back(key);
    } else {
      slot = slot_of[key] - 1;
    }
    pair_slot.push_back(slot);
    pair_right.push_back(pack_tag(ri, rj));
    return true;
  }

  // PermutationBuilder::build (lib.rs:62-93): merge the cycles of `left` and `right` (smaller into larger),
  // relabel the smaller cycle, then swap the two successors.  Consumes the constraints like `mem::take`.
  // Returns false when a tag does not fit `size` rows (the reference would index out of bounds and panic).
  bool build(size_t size, uint64_t* mapping) {
    const size_t len = size * kColumns;
    std::vector<uint32_t> start(keys.size() + 1, 0);
    for (uint32_t s : pair_slot) start[s + 1]++;
    for (size_t k = 0; k < keys.size(); k++) start[k + 1] += start[k];
    std::vector<uint64_t> grouped(pair_right.size());
    {
      std::vector<uint32_t> fill(start.begin(), start.end() - 1);
      for (size_t p = 0; p < pair_slot.size(); p++) grouped[fill[pair_slot[p]]++] = pair_right[p];
    }
    bool ok = true;
    for (uint64_t t : keys) ok &= tag_col(t) < kColumns && tag_row(t) < size;
    for (uint64_t t : pair_right) ok &= tag_col(t) < kColumns && tag_row(t) < size;
    if (ok) {
      std::vector<uint64_t> aux(len), sizes(len, 1);
      for (size_t k = 0; k < len; k++) mapping[k] = aux[k] = k;
      for (size_t c = 0; c < keys.size(); c++) {
        uint64_t left = tag_row(keys[c]) + tag_col(keys[c]) * size;
        for (uint32_t p = start[c]; p < start[c + 1]; p++) {
          uint64_t right = tag_row(grouped[p]) + tag_col(grouped[p]) * size;
          if (aux[left] == aux[right]) continue;
          if (sizes[aux[left]] < sizes[aux[right]]) std::swap(left, right);
          sizes[aux[left]] += sizes[aux[right]];
          const uint64_t label = aux[left];
          uint64_t next = right;
          do {
            aux[next] = label;
            next = mapping[next];
          } while (aux[next] != label);
          std::swap(mapping[left], mapping[right]);
        }
      }
    }
    slot_of.clear();
    keys.clear();
    pair_slot.clear();
    pair_right.clear();
    return ok;
  }
};

}  // namespace

struct tp_permutation_builder {
  CopyConstraints cc;
};

struct tp_trace {
  size_t n_inputs = 0;
  uint64_t next_var = 0;             // Context::new_id, builder.rs:132-139
  std::vector<uint8_t> kind;         // per gate: TP_GATE_MUL / TP_GATE_ADD
  std::vector<uint64_t> lhs, rhs;    // per gate: VALUE slots of the operands (see value_slot)
  std::vector<uint64_t> tag_of;      // var id -> packed tag or kNoTag   (InnerContext::var_map)
  std::vector<uint64_t> value_slot;  // var id -> value slot: input k -> k, output of gate j -> n_inputs + j,
                                     // a copy id made for an already-placed operand -> its source's slot
  std::vector<uint64_t> pending_l, pending_r;  // InnerContext::pending_eq
  CopyConstraints cc;
  bool finished = false;
  size_t rows = 0;

  uint64_t new_id(uint64_t slot) {
    tag_of.push_back(kNoTag);
    value_slot.push_back(slot);
    return next_var++;
  }
  // Context::add_eq (builder.rs:148-166): both placed -> a copy constraint, else remembered until finish().
  bool add_eq(uint64_t l, uint64_t r) {
    uint64_t a = tag_of[l], b = tag_of[r];
    if (a != kNoTag && b != kNoTag) return cc.add(tag_col(a), tag_row(a), tag_col(b), tag_row(b));
    pending_l.push_back(l);
    pending_r.push_back(r);
    return true;
  }
};

#define TP_TRY_ALLOC(stmt)          \
  try {                             \
    stmt;                           \
  } catch (const std::bad_alloc&) { \
    return TP_ERR_INVALID_ARG;      \
  }

#define TP_TRY_OK(stmt)             \
  do {                              \
    int rc__ = (stmt);              \
    if (rc__ != TP_OK) return rc__; \
  } while (0)

extern "C" {

// ---- Fr conversions for host languages without a big-integer type (the C++ mirror, include/typlonk_b200.hpp) -------

// Fr::from(i64): negative values map to r - |v| (ark-ff `From<i32/i64>`, used by plonk/src/utils.rs:152-153)
int tp_fr_from_i64(int64_t v, uint64_t out[4]) {
  if (!out) return TP_ERR_INVALID_ARG;
  const uint64_t mag = v < 0 ? (uint64_t)0 - (uint64_t)v : (uint64_t)v;
  HFr x = HFr::from_u64(mag);
  if (v < 0) x = x.neg();
  memcpy(out, x.v, 32);
  return TP_OK;
}
// 32-byte little-endian canonical integer (< r, else TP_ERR_MALFORMED) <-> Montgomery limbs
int tp_fr_from_canonical(const uint8_t in[32], uint64_t out[4]) {
  if (!in || !out) return TP_ERR_INVALID_ARG;
  uint64_t v[4];
  memcpy(v, in, 32);
  if (tph::ge<4>(v, tph::FR_PARAMS.mod)) return TP_ERR_MALFORMED;
  HFr m = HFr::to_mont(v);
  memcpy(out, m.v, 32);
  return TP_OK;
}
int tp_fr_to_canonical(const uint64_t in[4], uint8_t out[32]) {
  if (!in || !out) return TP_ERR_INVALID_ARG;
  HFr m;
  memcpy(m.v, in, 32);
  if (tph::ge<4>(m.v, tph::FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  HFr c = m.from_mont();
  memcpy(out, c.v, 32);
  return TP_OK;
}

// ---- the permutation crate's builder on its own ---------------------------------------------------------------

int tp_permutation_builder_create(size_t rows, tp_permutation_builder** out) {
  if (!out) return TP_ERR_INVALID_ARG;
  tp_permutation_builder* b = new (std::nothrow) tp_permutation_builder();
  if (!b) return TP_ERR_INVALID_ARG;
  b->cc.rows = rows;
  *out = b;
  return TP_OK;
}
int tp_permutation_builder_destroy(tp_permutation_builder* b) {
  delete b;
  return TP_OK;
}
int tp_permutation_builder_add_row(tp_permutation_builder* b) {
  if (!b) return TP_ERR_INVALID_ARG;
  b->cc.rows++;
  return TP_OK;
}
int tp_permutation_builder_add_constrain(tp_permutation_builder* b, size_t left_i, size_t left_j, size_t right_i,
                                         size_t right_j) {
  if (!b) return TP_ERR_INVALID_ARG;
  TP_TRY_ALLOC(if (!b->cc.add(left_i, left_j, right_i, right_j)) return TP_ERR_INVALID_TAG)
  return TP_OK;
}
int tp_permutation_builder_build(tp_permutation_builder* b, size_t size, uint64_t* perm) {
  if (!b || !perm || size == 0) return TP_ERR_INVALID_ARG;
  TP_TRY_ALLOC(if (!b->cc.build(size, perm)) return TP_ERR_INVALID_TAG)
  return TP_OK;
}

// ---- circuit tracing ------------------------------------------------------------------------------------------

int tp_trace_create(size_t n_inputs, tp_trace** out) {
  if (!out) return TP_ERR_INVALID_ARG;
  tp_trace* t = new (std::nothrow) tp_trace();
  if (!t) return TP_ERR_INVALID_ARG;
  t->n_inputs = n_inputs;
  TP_TRY_ALLOC(for (size_t k = 0; k < n_inputs; k++) t->new_id(k))  // BuildVar::input, builder.rs:371-377
  *out = t;
  return TP_OK;
}

int tp_trace_create_public(size_t n_inputs, size_t n_public, tp_trace** out) {
  if (!out || n_public > n_inputs) return TP_ERR_INVALID_ARG;
  TP_TRY_OK(tp_trace_create(n_inputs, out));
  tp_trace* t = *out;
  // public gate j = input j at (0, j); its output slot n_inputs + j exists but no variable refers to it
  TP_TRY_ALLOC(for (size_t j = 0; j < n_public; j++) {
    t->kind.push_back(TP_GATE_PUBLIC);
    t->lhs.push_back(j);
    t->rhs.push_back(j);
    t->cc.rows++;
    t->tag_of[j] = pack_tag(0, j);
  })
  return TP_OK;
}

int tp_trace_destroy(tp_trace* t) {
  delete t;
  return TP_OK;
}

static int trace_gate(tp_trace* t, int kind, uint64_t l, uint64_t r, uint64_t* out_var) {
  if (t->finished) return TP_ERR_INVALID_ARG;
  if (kind != TP_GATE_MUL && kind != TP_GATE_ADD) return TP_ERR_INVALID_ARG;
  if (l >= t->next_var || r >= t->next_var) return TP_ERR_INVALID_ARG;
  // builder.rs:339-370.  add_gate first (the row exists before its tags are checked), then the output id, then the
  // two operands in order: an operand already placed in a cell gets a fresh id in this row and an equality with the
  // old one; an operand seen for the first time is placed here.
  const uint64_t j = t->kind.size();
  t->kind.push_back((uint8_t)kind);
  t->lhs.push_back(t->value_slot[l]);
  t->rhs.push_back(t->value_slot[r]);
  t->cc.rows++;
  const uint64_t out = t->new_id(t->n_inputs + j);
  t->tag_of[out] = pack_tag(2, j);
  const uint64_t ids[2] = {l, r};
  for (uint64_t i = 0; i < 2; i++) {
    const uint64_t id = ids[i];
    if (t->tag_of[id] != kNoTag) {
      const uint64_t copy = t->new_id(t->value_slot[id]);
      t->tag_of[copy] = pack_tag(i, j);
      if (!t->add_eq(id, copy)) return TP_ERR_INVALID_TAG;
    } else {
      t->tag_of[id] = pack_tag(i, j);
    }
  }
  if (out_var) *out_var = out;
  return TP_OK;
}

int tp_trace_gate(tp_trace* t, int kind, uint64_t lhs, uint64_t rhs, uint64_t* out_var) {
  if (!t) return TP_ERR_INVALID_ARG;
  TP_TRY_ALLOC(return trace_gate(t, kind, lhs, rhs, out_var))
}

int tp_trace_gates(tp_trace* t, size_t count, const uint8_t* kinds, const uint64_t* lhs, const uint64_t* rhs,
                   uint64_t* out_vars) {
  if (!t || (count && (!kinds || !lhs || !rhs))) return TP_ERR_INVALID_ARG;
  for (size_t k = 0; k < count; k++) {
    uint64_t out = 0;
    int rc;
    TP_TRY_ALLOC(rc = trace_gate(t, kinds[k], lhs[k], rhs[k], &out))
    if (rc != TP_OK) return rc;
    if (out_vars) out_vars[k] = out;
  }
  return TP_OK;
}

int tp_trace_assert_eq(tp_trace* t, uint64_t a, uint64_t b) {
  if (!t || t->finished || a >= t->next_var || b >= t->next_var) return TP_ERR_INVALID_ARG;
  TP_TRY_ALLOC(if (!t->add_eq(a, b)) return TP_ERR_INVALID_TAG)  // BuildVar::assert_eq, builder.rs:427-433
  return TP_OK;
}

int tp_trace_finish(tp_trace* t, size_t* rows, size_t* gates) {
  if (!t) return TP_ERR_INVALID_ARG;
  if (!t->finished) {
    // Context::finish, builder.rs:167-186: retry the parked equalities once, all must resolve now
    std::vector<uint64_t> pl, pr;
    pl.swap(t->pending_l);
    pr.swap(t->pending_r);
    for (size_t k = 0; k < pl.size(); k++) TP_TRY_ALLOC(if (!t->add_eq(pl[k], pr[k])) return TP_ERR_INVALID_TAG)
    if (!t->pending_l.empty()) return TP_ERR_UNPLACED_VARIABLE;  // assert!(inner.pending_eq.is_empty())
    size_t size = 2;                                             // fill(), builder.rs:47-58
    while (size < t->kind.size() + 3) size *= 2;
    t->rows = size;
    t->finished = true;
  }
  if (rows) *rows = t->rows;
  if (gates) *gates = t->kind.size();
  return TP_OK;
}

int tp_trace_gate_kinds(const tp_trace* t, uint8_t* out) {
  if (!t || !t->finished || !out) return TP_ERR_INVALID_ARG;
  memcpy(out, t->kind.data(), t->kind.size());
  memset(out + t->kind.size(), TP_GATE_DUMMY, t->rows - t->kind.size());
  return TP_OK;
}

// Selector columns as evaluations over the domain, [q_l | q_r | q_o | q_m | q_c], each `rows` Fr in Montgomery form
// (builder.rs:73-84 transposes Gate::to_row the same way): Mul = [0,0,1,1,0], Add = [1,1,1,0,0], Dummy = 0,
// Public = [1,0,0,0,0].
int tp_trace_selectors(const tp_trace* t, uint64_t* out) {
  if (!t || !t->finished || !out) return TP_ERR_INVALID_ARG;
  const size_t n = t->rows;
  memset(out, 0, 5 * n * 32);
  const HFr one = HFr::one();
  for (size_t j = 0; j < t->kind.size(); j++) {
    if (t->kind[j] == TP_GATE_PUBLIC) {   // q_l = 1 only: x_i + PI_i = 0
      memcpy(out + j * 4, one.v, 32);
      continue;
    }
    const bool mul = t->kind[j] == TP_GATE_MUL;
    memcpy(out + (2 * n + j) * 4, one.v, 32);
    if (mul) {
      memcpy(out + (3 * n + j) * 4, one.v, 32);
    } else {
      memcpy(out + (0 * n + j) * 4, one.v, 32);
      memcpy(out + (1 * n + j) * 4, one.v, 32);
    }
  }
  return TP_OK;
}

int tp_trace_permutation(tp_trace* t, uint64_t* perm) {
  if (!t || !t->finished || !perm) return TP_ERR_INVALID_ARG;
  TP_TRY_ALLOC(if (!t->cc.build(t->rows, perm)) return TP_ERR_INVALID_TAG)
  return TP_OK;
}

// CompiledCircuit::prove's witness part (proof.rs:33-49): replay the gates over Fr (ComputeVar::binary_operation,
// builder.rs:380-397, pushes left | right | value per gate), zero-fill to rows - 3, append three blinders per column.
// `blinders` = a0 a1 a2 b0 b1 b2 c0 c1 c2 (the order the reference draws them in).
int tp_trace_witness(const tp_trace* t, const uint64_t* inputs, size_t n_inputs, const uint64_t* blinders,
                     uint64_t* const advice[3]) {
  if (!t || !t->finished || !blinders || !advice || n_inputs != t->n_inputs || (n_inputs && !inputs))
    return TP_ERR_INVALID_ARG;
  for (int k = 0; k < 3; k++)
    if (!advice[k]) return TP_ERR_INVALID_ARG;
  const size_t n = t->rows, g = t->kind.size();
  for (int k = 0; k < 9; k++)
    if (tph::ge<4>(blinders + 4 * k, tph::FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;  // not a field element
  std::vector<HFr> val;
  TP_TRY_ALLOC(val.resize(n_inputs + g))
  for (size_t k = 0; k < n_inputs; k++) {
    memcpy(val[k].v, inputs + 4 * k, 32);
    if (tph::ge<4>(val[k].v, tph::FR_PARAMS.mod)) return TP_ERR_INVALID_ARG;
  }
  HFr* a = reinterpret_cast<HFr*>(advice[0]);
  HFr* b = reinterpret_cast<HFr*>(advice[1]);
  HFr* c = reinterpret_cast<HFr*>(advice[2]);
  for (size_t j = 0; j < g; j++) {
    const HFr l = val[t->lhs[j]], r = val[t->rhs[j]];
    if (t->kind[j] == TP_GATE_PUBLIC) {   // a = x_i, b = c = 0
      a[j] = l;
      b[j] = c[j] = val[n_inputs + j] = HFr::zero();
      continue;
    }
    const HFr v = t->kind[j] == TP_GATE_MUL ? l * r : l + r;
    val[n_inputs + j] = v;
    a[j] = l;
    b[j] = r;
    c[j] = v;
  }
  for (int k = 0; k < 3; k++) {
    memset(advice[k] + 4 * g, 0, (n - 3 - g) * 32);
    memcpy(advice[k] + 4 * (n - 3), blinders + 12 * k, 96);
  }
  return TP_OK;
}

}  // extern "C"
