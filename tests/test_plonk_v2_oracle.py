"""CPU tests of proof format v2 (DESIGN.md, "Proof format v2"): the oracle's prover and verifier, the forgery v1
admits and v2 does not, the tracer's public gates against a restatement, the key layout, and the library's host-only
verifier and decoders on oracle-made proofs."""
import pytest

from oracle.pyoracle import builder as ob, plonk as oplonk, plonk_v2 as ov2, rng
from oracle.pyoracle.curve import g1_deserialize_unchecked
from oracle.pyoracle.fields import R_MOD, fr_to_mont

import forge_v1

TAU = rng.fr_rand_stream(1, 1)[0]
BLINDERS = rng.fr_rand_stream(2, 9)

# (circuit, inputs count, inputs, l) -> n = 8, 8, 16, 64, 256
CASES = [("readme", ob.circuit_pythagoras, 3, [3, 4, 5], 0),
         ("readme", ob.circuit_pythagoras, 3, [3, 4, 5], 1),
         ("readme", ob.circuit_pythagoras, 3, [3, 4, 5], 2),
         ("mul40", ob.make_mul_chain(40), 2, [3, 5], 1),
         ("mul200", ob.make_mul_chain(200), 2, [3, 5], 2)]


@pytest.fixture(scope="module", params=CASES, ids=lambda c: "%s-l%d" % (c[0], c[4]))
def made(request):
    _, run, n_inputs, inputs, ell = request.param
    circuit = ov2.compile_circuit(run, n_inputs, ell, TAU)
    return circuit, ov2.vk_bytes(circuit), ov2.prove(circuit, inputs, BLINDERS)


def test_oracle_accepts_its_own_proofs(made):
    circuit, vk, proof = made
    assert circuit.oc.domain.size in (8, 16, 64, 256)
    assert len(proof.block()) == ov2.PROOF_BYTES
    assert ov2.verify(vk, circuit.oc.srs, proof, proof.public_values, use_trapdoor=True)


def test_oracle_pairing_verifier_agrees():
    circuit = ov2.compile_circuit(ob.circuit_pythagoras, 3, 1, TAU)
    vk = ov2.vk_bytes(circuit)
    proof = ov2.prove(circuit, [3, 4, 5], BLINDERS)
    assert ov2.verify(vk, circuit.oc.srs, proof, proof.public_values)
    bad = ov2.ProofV2(proof.points, proof.evals[:5] + [(proof.evals[5] + 1) % R_MOD], proof.public_values)
    assert not ov2.verify(vk, circuit.oc.srs, bad, bad.public_values)


def _corruptions(proof):
    for i in range(9):
        pts = list(proof.points)
        pts[i] = pts[(i + 1) % 9]
        yield ov2.ProofV2(pts, proof.evals, proof.public_values)
    for i in range(6):
        evs = list(proof.evals)
        evs[i] = (evs[i] + 1) % R_MOD
        yield ov2.ProofV2(proof.points, evs, proof.public_values)


def test_oracle_rejects_each_corrupted_field(made):
    circuit, vk, proof = made
    for bad in _corruptions(proof):
        assert not ov2.verify(vk, circuit.oc.srs, bad, bad.public_values, use_trapdoor=True)


def test_oracle_rejects_wrong_public_values_count_and_key(made):
    circuit, vk, proof = made
    srs, pub = circuit.oc.srs, proof.public_values
    if pub:
        wrong = [(pub[0] + 1) % R_MOD] + pub[1:]
        assert not ov2.verify(vk, srs, ov2.ProofV2(proof.points, proof.evals, wrong), wrong, use_trapdoor=True)
    assert not ov2.verify(vk, srs, ov2.ProofV2(proof.points, proof.evals, pub + [0]), pub + [0], use_trapdoor=True)
    other = ov2.compile_circuit(ob.circuit_additive, 5, len(pub), TAU)
    assert not ov2.verify(ov2.vk_bytes(other), srs, proof, pub, use_trapdoor=True)


def test_public_gates_bind_the_statement():
    """A proof for public c = 5 does not verify as one for c = 6, and the prover reads c from the witness."""
    circuit = ov2.compile_circuit(ob.circuit_pythagoras, 3, 3, TAU)
    vk = ov2.vk_bytes(circuit)
    proof = ov2.prove(circuit, [3, 4, 5], BLINDERS)
    assert proof.public_values == [3, 4, 5]
    assert ov2.verify(vk, circuit.oc.srs, proof, [3, 4, 5], use_trapdoor=True)
    assert not ov2.verify(vk, circuit.oc.srs, ov2.ProofV2(proof.points, proof.evals, [3, 4, 6]), [3, 4, 6],
                          use_trapdoor=True)


def test_v1_forgery_is_accepted_by_the_v1_verifier():
    """Records the defect of v1: a proof of 3^2 + 4^2 = 6^2."""
    oc, pf = forge_v1.forged_v1_proof(TAU, BLINDERS)
    assert pf.r[1] == 0
    assert oplonk.verify(oc, pf, use_trapdoor=True)
    assert oplonk.verify(oc, pf)
    with pytest.raises(oplonk.GateUnsatisfied.__mro__[1]):   # the honest prover cannot make one
        honest = oplonk.prove(oc, forge_v1.FALSE_INPUTS, [0], BLINDERS)
        assert oplonk.verify(oc, honest, use_trapdoor=True)


@pytest.mark.parametrize("ell", [0, 1])
def test_same_forgery_fails_against_v2(ell):
    circuit, vk, proof = forge_v1.forged_v2_attempt(TAU, BLINDERS, ell)
    assert not ov2.verify(vk, circuit.oc.srs, proof, proof.public_values, use_trapdoor=True)


# ---- the tracer's public gates: library vs a restatement -------------------------------------------------------

@pytest.mark.parametrize("n_public", [0, 1, 2, 3])
def test_native_public_gates_match_the_restatement(n_public):
    from typlonk_b200 import field as F
    from typlonk_b200.ffi import Trace
    from typlonk_b200.plonk import TraceVar, KIND_NAMES
    t = Trace(3, n_public)
    ob.circuit_pythagoras([TraceVar(t, k) for k in range(3)])
    rows, _ = t.finish()
    gates, perm = ov2.trace_public(ob.circuit_pythagoras, 3, n_public)
    assert rows == len(gates)
    assert [KIND_NAMES[k] for k in t.gate_kinds()] == gates
    sel = bytes(t.selectors())
    for k in range(5):
        assert F.fr_vec_from_bytes(sel[k * rows * 32:(k + 1) * rows * 32]) == [ov2.ROWS[g][k] for g in gates]
    import struct
    native = list(struct.unpack("<%dQ" % (3 * rows), bytes(t.permutation())))
    assert native == list(perm.perm)
    cols = t.witness(F.fr_vec_to_bytes([3, 4, 5]), F.fr_vec_to_bytes(BLINDERS))
    oc = ov2.CircuitV2(type("C", (), {"rows": rows, "run": staticmethod(ob.circuit_pythagoras)})(), n_public)
    want = ov2.witness_columns(oc, [3, 4, 5], BLINDERS)
    for k in range(3):
        assert F.fr_vec_from_bytes(bytes(cols[k])) == want[k]


def test_native_tracer_refuses_public_kind_and_bad_count():
    from typlonk_b200.ffi import Trace, TyplonkError
    with pytest.raises(TyplonkError):
        Trace(2, 3)
    t = Trace(2, 1)
    with pytest.raises(TyplonkError):
        t.gate(3, 0, 1)


# ---- the key layout and the host-only verifier -------------------------------------------------------------------

def test_vk2_layout_and_size():
    circuit = ov2.compile_circuit(ob.circuit_pythagoras, 3, 2, TAU)
    raw = ov2.vk_bytes(circuit)
    assert len(raw) == 1368 == 4 + 4 + 8 + 8 + 3 * 32 + 9 * 96 + 2 * 192
    assert raw[:4] == b"TPK2" and int.from_bytes(raw[4:8], "little") == 1
    assert int.from_bytes(raw[8:16], "little") == circuit.oc.domain.size
    assert int.from_bytes(raw[16:24], "little") == 2
    assert [int.from_bytes(raw[24 + 32 * i: 56 + 32 * i], "little") for i in range(3)] == list(circuit.oc.copy_constrains.cosets)
    pts = [g1_deserialize_unchecked(raw[120 + 96 * i: 216 + 96 * i]) for i in range(9)]
    assert pts[:5] == list(circuit.oc.fixed_commitments)
    assert pts[5:8] == ov2.sigma_commitments(circuit.oc)
    assert raw[984:1176] == ov2.g2_wire(circuit.oc.srs.g2) and raw[1176:] == ov2.g2_wire(circuit.oc.srs.g2s)


def _mont(vals):
    return b"".join(fr_to_mont(v % R_MOD).to_bytes(32, "little") for v in vals)


def test_host_verifier_agrees_with_the_oracle(made):
    from typlonk_b200.plonk import ProofV2, VerifyingKeyV2
    circuit, vk, proof = made
    key = VerifyingKeyV2.from_bytes(vk)
    assert key.to_bytes() == vk
    mine = ProofV2(proof.block(), proof.public_values)
    assert key.verify(mine)
    assert ProofV2.from_bytes(proof.to_bytes()) == mine
    for bad in _corruptions(proof):
        assert not key.verify(ProofV2(bad.block(), bad.public_values))
    if proof.public_values:
        assert not key.verify(mine, [(proof.public_values[0] + 1) % R_MOD] + proof.public_values[1:])
    assert not key.verify(mine, proof.public_values + [0])
    forged = forge_v1.forged_v2_attempt(TAU, BLINDERS, 0)
    assert not VerifyingKeyV2.from_bytes(forged[1]).verify(ProofV2(forged[2].block(), []))
