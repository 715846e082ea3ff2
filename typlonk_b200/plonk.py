"""Host-side mirror of the reference's `plonk` crate API over the CUDA library:
CircuitDescription / Var (plonk/src/description.rs:4-16), CircuitBuilder::compile
(plonk/src/builder.rs:60-113), CompiledCircuit::prove (plonk/src/proof.rs:26-57).

    class Circuit(CircuitDescription):
        INPUTS = 3
        @staticmethod
        def run(inputs):
            a, b, c = inputs
            a = a.clone() * a; b = b.clone() * b; c = c.clone() * c
            d = a + b
            d.assert_eq(c)

    circuit = Circuit.build(ctx, tau)                 # description.rs:6-8
    proof = circuit.prove([3, 4, 5], [0], blinders)   # proof.rs:26

The circuit closure is run ONCE over `TraceVar`, which records every `+` / `*` / `assert_eq` into the
library's native tracer (csrc/trace.cpp, SURVEY.md 8 f3); padding, selector columns, the copy-constraint
permutation and every proof's witness columns come from that recording in C++ (the reference re-runs
the closure over ComputeVar for every proof, builder.rs:380-397); a Python restatement of that two-pass scheme,
which the CPU tests compare the native tracer with, lives in tests/py_tracer.py.  Everything numeric -- SRS, selector interpolation and commitments,
sigma tables, the whole prover -- runs on the device in libtyplonk_b200.  tau and the nine blinders are explicit inputs where the
reference draws them from thread_rng (builder.rs:71, proof.rs:42-48).  `verify` (proof.rs:59-63) runs
its circuit-sized parts on the device and the pairings on the host inside the library (csrc/verify.cu).
"""
import struct
from dataclasses import dataclass
from typing import List, Tuple

from . import field as F
from .ffi import (Context, GateUnsatisfied, TyplonkError, PROOF_FIXED_BYTES, GATE_ADD, GATE_MUL, Trace,  # noqa: F401
                  proof_decode, proof_decode_compressed, proof_encode, proof_encode_compressed)
from .kzg import Srs
from .permutation import Permutation

GATE_ROWS = {"Mul": (0, 0, 1, 1, 0), "Add": (1, 1, 1, 0, 0), "Dummy": (0, 0, 0, 0, 0)}  # builder.rs:318-324


class Var:
    """description.rs:10-16: `+`, `*`, `clone`, `assert_eq`."""

    def clone(self):
        raise NotImplementedError

    def assert_eq(self, other):
        raise NotImplementedError


class TraceVar(Var):
    """A variable of the native tracer: an id in a tp_trace (BuildVar, builder.rs:327-378, 427-433)."""

    def __init__(self, trace: Trace, vid: int):
        self.trace, self.id = trace, vid

    def clone(self):
        return TraceVar(self.trace, self.id)

    def __add__(self, rhs):
        return TraceVar(self.trace, self.trace.gate(GATE_ADD, self.id, rhs.id))

    def __mul__(self, rhs):
        return TraceVar(self.trace, self.trace.gate(GATE_MUL, self.id, rhs.id))

    def assert_eq(self, other):
        self.trace.assert_eq(self.id, other.id)


KIND_NAMES = {0: "Mul", 1: "Add", 2: "Dummy"}


@dataclass
class Proof:
    """proof.rs:85-95 as bytes: `fixed` is the 1472-byte block tp_prove writes, followed by the
    n-padded public inputs (u64 LE length + n x 32 B), SURVEY.md App. A.6."""
    fixed: bytes
    public_inputs: List[int]

    def to_bytes(self, compressed=False) -> bytes:
        """tp_proof_encode (the additive `Proof::to_bytes` of SURVEY.md 8 f4), or tp_proof_encode_compressed: the
        same framing with compressed points (an 848-byte block instead of 1472)."""
        encode = proof_encode_compressed if compressed else proof_encode
        return encode(self.fixed, F.fr_vec_to_bytes(self.public_inputs))

    @classmethod
    def from_bytes(cls, raw: bytes, compressed=False) -> "Proof":
        """tp_proof_decode: checked (canonical scalars and coordinates, points on the curve, exact length);
        raises ffi.Malformed otherwise.  compressed=True: tp_proof_decode_compressed, which recovers every y (an x
        without a root is malformed); `fixed` is the uncompressed block either way."""
        fixed, pis = (proof_decode_compressed if compressed else proof_decode)(raw)
        return cls(fixed, F.fr_vec_from_bytes(pis))


class CompiledCircuit:
    """plonk/src/lib.rs:18-26."""

    def __init__(self, desc, ctx, srs, handle, rows, fixed_commitments, gates, perm, native_trace):
        self.desc, self.ctx, self.srs, self.handle = desc, ctx, srs, handle
        self.rows = rows
        self.fixed_commitments = fixed_commitments
        self.gates = gates
        self.perm = perm
        self.native_trace = native_trace

    def witness_bytes(self, inputs, blinders):
        """proof.rs:33-49 through tp_trace_witness: three columns of rows x 32 B Montgomery limbs."""
        assert len(blinders) == 9
        return self.native_trace.witness(F.fr_vec_to_bytes(inputs), F.fr_vec_to_bytes(blinders))

    def prove(self, inputs, public_inputs, blinders) -> Proof:
        """CompiledCircuit::prove (proof.rs:26-57).  Raises GateUnsatisfied where the reference
        panics in `vanishes`."""
        cols = self.witness_bytes(inputs, blinders)
        given = [v % F.R_MOD for v in public_inputs][: self.rows]
        pis = (given + [0] * self.rows)[: self.rows]          # what Proof.public_inputs carries (proof.rs:52-53, 190)
        fixed = self.handle.prove_inputs(cols, F.fr_vec_to_bytes(given))
        return Proof(fixed, pis)

    def prove_batch(self, inputs_list, public_inputs_list, blinders_list) -> List[Proof]:
        """Many proofs of this circuit in one call (tp_prove_batch); proof k equals prove(inputs_list[k],
        public_inputs_list[k], blinders_list[k]).  Raises what prove would raise for the first failing proof, naming
        its index."""
        count = len(inputs_list)
        assert len(public_inputs_list) == count and len(blinders_list) == count
        cols = [self.witness_bytes(i, b) for i, b in zip(inputs_list, blinders_list)]
        given = [[v % F.R_MOD for v in pi][: self.rows] for pi in public_inputs_list]
        fixed, status = self.handle.prove_batch(cols, [F.fr_vec_to_bytes(g) for g in given])
        for k, st in enumerate(status):
            if st == 6:
                raise GateUnsatisfied(st, "prove_batch: proof %d: gate constraints do not vanish on the domain" % k)
            if st != 0:
                raise TyplonkError(st, "prove_batch: proof %d: permutation prove: zero denominator" % k)
        return [Proof(f, (g + [0] * self.rows)[: self.rows]) for f, g in zip(fixed, given)]

    def verify(self, proof: Proof) -> bool:
        """CompiledCircuit::verify (proof.rs:59-63, 195-233)."""
        return self.handle.verify(proof.fixed, F.fr_vec_to_bytes(proof.public_inputs))

    def verify_batch(self, proofs: List[Proof]):
        """Every proof of this circuit checked at once (tp_verify_batch): (all accepted, per-proof verdicts).  Stricter
        than `verify` on points outside the prime-order subgroup, which it rejects."""
        return self.handle.verify_batch([p.fixed for p in proofs], [F.fr_vec_to_bytes(p.public_inputs) for p in proofs])

    def verifying_key(self) -> "VerifyingKey":
        """What `verify` reads of this circuit, without the prover's state (tp_vk_from_circuit); it stays valid after
        the circuit is destroyed."""
        return VerifyingKey(self.handle.verifying_key())


class VerifyingKey:
    """A verification key: n, the coset representatives, the eight circuit commitments, srs[0], the SRS's two G2
    points and sigma_1, sigma_2 in coefficient form (the proof does not carry their values at the challenge point), so
    1376 + 64n bytes on the wire."""

    def __init__(self, handle):
        self.handle = handle

    @property
    def ctx(self):
        return self.handle.ctx

    def to_bytes(self) -> bytes:
        """tp_vk_serialize."""
        return bytes(self.handle.serialize())

    @classmethod
    def from_bytes(cls, ctx: Context, raw: bytes, check=2) -> "VerifyingKey":
        """tp_vk_deserialize (check 0: encoding and framing, 1: + on the curve, 2: + prime-order subgroups); raises
        ffi.Malformed naming the rejected field."""
        return cls(ctx.vk_deserialize(raw, check))

    def verify(self, proof: Proof) -> bool:
        """CompiledCircuit::verify against the key (tp_vk_verify): the verdict `CompiledCircuit.verify` gives."""
        return self.handle.verify(proof.fixed, F.fr_vec_to_bytes(proof.public_inputs))


def verify_batch(pairs: List[Tuple[VerifyingKey, Proof]]) -> Tuple[bool, List[bool]]:
    """Proofs of several circuits in one folded check (tp_vk_verify_batch): (all accepted, per-proof verdicts).  Every
    key must belong to one context; keys of different sizes and SRSes may be mixed."""
    if not pairs:
        return True, []
    keys, key_of, index = [], [], {}
    for vk, _ in pairs:
        if id(vk.handle) not in index:
            index[id(vk.handle)] = len(keys)
            keys.append(vk.handle)
        key_of.append(index[id(vk.handle)])
    ctx = keys[0].ctx
    return ctx.vk_verify_batch(keys, key_of, [p.fixed for _, p in pairs],
                               [F.fr_vec_to_bytes(p.public_inputs) for _, p in pairs])


class CircuitDescription:
    """description.rs:4-9."""
    INPUTS = 0

    @staticmethod
    def run(inputs):
        raise NotImplementedError

    @classmethod
    def trace_native(cls) -> Trace:
        """The closure recorded once by the library's tracer (finished: padded, equalities resolved)."""
        t = Trace(cls.INPUTS)
        cls.run([TraceVar(t, k) for k in range(cls.INPUTS)])
        t.finish()
        return t

    @classmethod
    def build(cls, ctx: Context, tau: int) -> CompiledCircuit:
        """CircuitBuilder::compile (builder.rs:60-113) with the SRS secret as an input."""
        t = cls.trace_native()
        rows = t.rows
        srs = Srs.from_secret(ctx, tau, rows)
        sel_all = t.selectors()
        sel = [bytes(sel_all[k * rows * 32:(k + 1) * rows * 32]) for k in range(5)]
        perm_bytes = bytes(t.permutation())
        handle, fixed = ctx.circuit_compile(srs.handle, sel, perm_bytes, rows)
        gates = [KIND_NAMES[k] for k in t.gate_kinds()]
        perm = Permutation(list(struct.unpack("<%dQ" % (3 * rows), perm_bytes)))
        return CompiledCircuit(cls, ctx, srs, handle, rows, [F.g1_from_abi(c) for c in fixed], gates, perm, t)
