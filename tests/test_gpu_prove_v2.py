"""GPU tests of proof format v2 (tp_prove_v2, tp_vk2_*, tp_verify_v2) against the v2 oracle
(oracle/pyoracle/plonk_v2.py): proof and key bytes equal under fixed tau / blinders, the host verifier and the oracle's
verifier accept, every corruption is rejected, and v1's forged proof is accepted by tp_verify, as documented."""
import os
import subprocess

import pytest

from oracle.pyoracle import builder as obuilder, plonk_v2 as ov2
from oracle.pyoracle.fields import R_MOD
from typlonk_b200.ffi import Context, GateUnsatisfied, Malformed, TyplonkError
from typlonk_b200.plonk import ProofV2, VerifyingKeyV2

from test_gpu_prove import Additive, Pythagoras, mul_chain, BLINDERS, TAU

pytestmark = pytest.mark.gpu


def public(desc, ell):
    class D(desc):
        PUBLIC = ell
    return D


CASES = [("readme", Pythagoras, obuilder.circuit_pythagoras, 3, [3, 4, 5]),
         ("additive", Additive, obuilder.circuit_additive, 5, [1, 2, 3, 4, -4]),
         ("mul5", mul_chain(5), obuilder.make_mul_chain(5), 2, [3, 5]),
         ("mul13", mul_chain(13), obuilder.make_mul_chain(13), 2, [3, 5]),
         ("mul61", mul_chain(61), obuilder.make_mul_chain(61), 2, [3, 5]),
         ("mul253", mul_chain(253), obuilder.make_mul_chain(253), 2, [3, 5])]

# one byte in each field of the 1056-byte block: the nine points, then the six evaluations
CORRUPTIONS = [96 * i + 7 for i in range(9)] + [864 + 32 * i + 3 for i in range(6)]


# every circuit at l = 0, 1, 2, and the README circuit with a, b and c public
PARAMS = [pytest.param(*c, ell, id="%s-l%d" % (c[0], ell)) for c in CASES for ell in (0, 1, 2)] + \
    [pytest.param(*CASES[0], 3, id="readme-l3")]


@pytest.mark.parametrize("name,desc,run,n_inputs,inputs,ell", PARAMS)
def test_bytes_equal_the_oracle(ctx, name, desc, run, n_inputs, inputs, ell):
    circuit = public(desc, ell).build(ctx, TAU)
    vk = circuit.verifying_key_v2()
    proof = circuit.prove_v2(inputs, BLINDERS)
    oc = ov2.compile_circuit(run, n_inputs, ell, TAU)
    ovk = ov2.vk_bytes(oc)
    assert vk.to_bytes() == ovk
    oproof = ov2.prove(oc, inputs, BLINDERS)
    assert proof.fixed == oproof.block()
    assert proof.to_bytes() == oproof.to_bytes()
    assert proof.public_inputs == [v % R_MOD for v in inputs[:ell]]
    assert vk.verify(proof)
    assert ov2.verify(ovk, oc.oc.srs, oproof, oproof.public_values, use_trapdoor=True)
    if name == "readme":
        assert ov2.verify(ovk, oc.oc.srs, oproof, oproof.public_values)   # the pairing form, once
    if ell:
        wrong = list(proof.public_inputs)
        wrong[0] = (wrong[0] + 1) % R_MOD
        assert not vk.verify(proof, wrong)


@pytest.fixture(scope="module")
def readme_c(ctx):
    circuit = public(Pythagoras, 1).build(ctx, TAU)
    return circuit, circuit.prove_v2([3, 4, 5], BLINDERS)


@pytest.mark.parametrize("off", CORRUPTIONS)
def test_every_corruption_is_rejected(readme_c, off):
    circuit, proof = readme_c
    vk = circuit.verifying_key_v2()
    assert vk.verify(proof)
    bad = bytearray(proof.fixed)
    bad[off] ^= 1
    assert not vk.verify(ProofV2(bytes(bad), proof.public_inputs))


@pytest.mark.parametrize("i", range(9))
def test_valid_point_in_the_wrong_place_is_rejected(readme_c, i):
    """Point i replaced by point i + 1 of the same proof: on the curve and in G1, so the pairing check decides."""
    circuit, proof = readme_c
    bad = bytearray(proof.fixed)
    j = (i + 1) % 9
    bad[96 * i: 96 * i + 96] = proof.fixed[96 * j: 96 * j + 96]
    assert not circuit.verifying_key_v2().verify(ProofV2(bytes(bad), proof.public_inputs))


def test_key_must_name_the_traced_public_count(ctx, readme_c):
    circuit, _ = readme_c   # traced with l = 1
    for ell in (0, 2):
        with pytest.raises(TyplonkError, match="public gate"):
            circuit.handle.verifying_key_v2(ell)


def test_wire_forms_round_trip_and_reject(readme_c):
    circuit, proof = readme_c
    vk = circuit.verifying_key_v2()
    raw = proof.to_bytes()
    assert len(raw) == 1056 + 8 + 32
    assert ProofV2.from_bytes(raw) == proof
    with pytest.raises(Malformed):
        ProofV2.from_bytes(raw[:-1])
    key = vk.to_bytes()
    for check in (0, 1, 2):
        again = VerifyingKeyV2.from_bytes(key, check)
        assert again.to_bytes() == key and again.verify(proof)
    bad = bytearray(key)
    bad[120 + 7] ^= 1   # q_l's x: off the curve (or not canonical)
    with pytest.raises(Malformed, match="q_l"):
        VerifyingKeyV2.from_bytes(bytes(bad), 1)
    with pytest.raises(Malformed, match="tag"):
        VerifyingKeyV2.from_bytes(b"TPVK" + key[4:], 0)


def test_wrong_key_wrong_count_and_other_circuit(ctx, readme_c):
    circuit, proof = readme_c
    other = public(Pythagoras, 2).build(ctx, TAU)
    assert not other.verifying_key_v2().verify(proof, proof.public_inputs + [0])
    assert not circuit.verifying_key_v2().verify(proof, [])
    chain = public(mul_chain(5), 1).build(ctx, TAU)
    assert not chain.verifying_key_v2().verify(proof)
    with pytest.raises(Exception):   # a key of another circuit is refused by the prover
        circuit.handle.prove_v2(chain.verifying_key_v2().handle, circuit.witness_bytes([3, 4, 5], BLINDERS), 1)


def test_key_outlives_circuit_and_context():
    c = Context(0)
    circuit = public(Pythagoras, 1).build(c, TAU)
    proof = circuit.prove_v2([3, 4, 5], BLINDERS)
    key = circuit.verifying_key_v2().to_bytes()
    c.close()
    assert VerifyingKeyV2.from_bytes(key).verify(proof)


def test_gate_and_copy_violations(ctx):
    circuit = public(Pythagoras, 1).build(ctx, TAU)
    vk = circuit.verifying_key_v2()
    cols = circuit.witness_bytes([3, 4, 5], BLINDERS)
    bad = [bytearray(c) for c in cols]
    bad[2][3 * 32] ^= 1                                 # c of gate 3 (a multiplication): the gate fails
    with pytest.raises(GateUnsatisfied):
        circuit.handle.prove_v2(vk.handle, bad, 1)
    # 3^2 + 4^2 != 6^2: every gate holds, the copy constraint d = c^2 does not
    fixed, pub = circuit.handle.prove_v2(vk.handle, circuit.witness_bytes([3, 4, 6], BLINDERS), 1)
    assert not vk.handle.verify(fixed, pub)


def test_device_group_gives_the_same_bytes(readme_c):
    _, proof = readme_c
    group = Context.multi([0, 0])
    gproof = public(Pythagoras, 1).build(group, TAU).prove_v2([3, 4, 5], BLINDERS)
    group.close()
    assert gproof == proof


@pytest.mark.parametrize("log_n", [16, 20])
def test_large_circuits_verify(ctx, log_n):
    gates = (1 << log_n) - 4
    circuit = public(mul_chain(gates), 1).build(ctx, TAU)
    assert circuit.rows == 1 << log_n
    proof = circuit.prove_v2([3, 5], BLINDERS)
    vk = circuit.verifying_key_v2()
    assert vk.verify(proof)
    bad = bytearray(proof.fixed)
    bad[864 + 1] ^= 1
    assert not vk.verify(ProofV2(bytes(bad), proof.public_inputs))
    # the oracle's trapdoor verifier is O(l): it checks the library's proof from the key bytes alone
    from oracle.pyoracle import kzg
    srs = kzg.Srs(None, None, None, secret=TAU % R_MOD)
    from oracle.pyoracle.curve import g1_deserialize_unchecked
    pts = [g1_deserialize_unchecked(proof.fixed[96 * i: 96 * i + 96]) for i in range(9)]
    evals = [int.from_bytes(proof.fixed[864 + 32 * i: 896 + 32 * i], "little") for i in range(6)]
    op = ov2.ProofV2(pts, evals, proof.public_inputs)
    assert ov2.verify(vk.to_bytes(), srs, op, proof.public_inputs, use_trapdoor=True)


def test_forged_v1_proof_is_accepted_by_tp_verify(ctx):
    """Records the v1 defect: t chosen after zeta makes r(zeta) = 0 for a false witness, and tp_verify accepts."""
    import forge_v1
    oc, pf = forge_v1.forged_v1_proof(TAU, BLINDERS)
    circuit = Pythagoras.build(ctx, TAU)
    assert circuit.handle.verify(pf.to_bytes()[:1472], bytes(32 * oc.rows))


def test_cpp_mirror(tmp_path):
    """tests/cpp/prove_v2_test.cpp: the whole v2 flow through include/typlonk_b200.hpp."""
    from typlonk_b200 import build
    build.build()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "typlonk_b200", "lib")
    exe = str(tmp_path / "prove_v2_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(root, "include"),
                          "-o", exe, os.path.join(root, "tests", "cpp", "prove_v2_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout, res.stdout + res.stderr
    assert "0 failures" in res.stdout
