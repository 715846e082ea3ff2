"""GPU tests of verification keys (tp_vk_* through plonk.VerifyingKey and plonk.verify_batch): the key's bytes against
the oracle restatement (tests/verify_key_ref.py), round trips at every check level, verdict parity with tp_verify
(corruptions, public inputs, a destroyed circuit), malformed keys, batches over several keys and SRSes, agreement with
tp_verify_batch, device groups, 2^16 and the C++ mirror."""
import os
import subprocess

import pytest

from oracle.pyoracle import builder as obuilder, rng
from oracle.pyoracle.fields import Q_MOD, R_MOD
from typlonk_b200.ffi import Context, Malformed, TyplonkError
from typlonk_b200.plonk import Proof, VerifyingKey, verify_batch

import verify_key_ref as ref
from test_gpu_prove import Additive, Pythagoras, mul_chain, BLINDERS, TAU
from test_gpu_verify_batch import CORRUPTIONS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAU2 = rng.fr_rand_stream(7, 1)[0]


def blinders(seed):
    return rng.fr_rand_stream(3000 + seed, 9)


def inputs_of(desc, k):
    if desc is Pythagoras:
        return [3, 4, 5]
    if desc is Additive:
        return [2 + k, 7, 2, 3 + k, 4]
    return [3 + k, 5 + 2 * k]


def proofs_of(circuit, count, seed=0):
    return [circuit.prove(inputs_of(circuit.desc, k), [0], blinders(seed + k)) for k in range(count)]


def corrupt(proof, off):
    bad = bytearray(proof.fixed)
    bad[off] ^= 1
    return Proof(bytes(bad), proof.public_inputs)


def outcome(fn, *args):
    """A verdict, or the error code where the call raises."""
    try:
        return bool(fn(*args))
    except TyplonkError as e:
        return ("error", e.code)


@pytest.fixture(scope="module")
def circuits(ctx):
    """README circuit, Additive, mul chains at 2^8, 2^10, 2^12 under TAU: (description, oracle run, inputs, circuit)."""
    out = {}
    for name, desc, run, n_in in (("readme", Pythagoras, obuilder.circuit_pythagoras, 3),
                                  ("additive", Additive, obuilder.circuit_additive, 5),
                                  ("chain8", mul_chain(253), obuilder.make_mul_chain(253), 2),
                                  ("chain10", mul_chain(1021), obuilder.make_mul_chain(1021), 2),
                                  ("chain12", mul_chain(4093), None, 2)):
        out[name] = (run, n_in, desc.build(ctx, TAU))
    return out


@pytest.mark.parametrize("name", ["readme", "additive", "chain8", "chain10"])
def test_key_bytes_equal_the_restatement_and_round_trip(ctx, circuits, name):
    run, n_in, circuit = circuits[name]
    raw = circuit.verifying_key().to_bytes()
    assert len(raw) == 1376 + 64 * circuit.rows
    assert raw == ref.vk_bytes(run, n_in, TAU)
    for check in (0, 1, 2):
        assert VerifyingKey.from_bytes(ctx, raw, check).to_bytes() == raw


@pytest.mark.parametrize("name", ["readme", "chain8"])
def test_single_verification_equals_tp_verify(ctx, circuits, name):
    _, _, circuit = circuits[name]
    vk = VerifyingKey.from_bytes(ctx, circuit.verifying_key().to_bytes())
    proofs = proofs_of(circuit, 2)
    for p in proofs:
        assert vk.verify(p) and circuit.verify(p)
    for off in CORRUPTIONS:
        bad = corrupt(proofs[0], off)
        assert outcome(vk.verify, bad) == outcome(circuit.verify, bad)
    # non-zero public inputs (the proof claims other public inputs than it was made with), reduced or not, too many
    pis = [5] + [0] * (circuit.rows - 1)
    claimed = Proof(proofs[1].fixed, pis)
    assert outcome(vk.verify, claimed) == outcome(circuit.verify, claimed) == False  # noqa: E712
    claimed = Proof(proofs[1].fixed, [0] * (circuit.rows - 1) + [R_MOD - 1])
    assert outcome(vk.verify, claimed) == outcome(circuit.verify, claimed) == False  # noqa: E712
    handle_pis = (R_MOD).to_bytes(32, "little")   # raw limbs >= r
    assert outcome(vk.handle.verify, proofs[1].fixed, handle_pis) == outcome(circuit.handle.verify, proofs[1].fixed, handle_pis)
    assert outcome(vk.handle.verify, proofs[1].fixed, bytes(32 * (circuit.rows + 1))) == ("error", 1)
    assert outcome(vk.handle.verify, proofs[1].fixed[:-1], b"") == outcome(circuit.handle.verify, proofs[1].fixed[:-1], b"")


def test_key_outlives_its_circuit(ctx):
    circuit = mul_chain(61).build(ctx, TAU)
    proofs = proofs_of(circuit, 2)
    vk = circuit.verifying_key()
    raw = vk.to_bytes()
    circuit.handle.destroy()
    assert vk.verify(proofs[0]) and vk.verify(proofs[1])
    assert not vk.verify(corrupt(proofs[0], 192))
    assert vk.to_bytes() == raw


def _expect_malformed(ctx, raw, check, words):
    with pytest.raises(Malformed) as e:
        ctx.vk_deserialize(bytes(raw), check)
    for w in words:
        assert w in str(e.value), str(e.value)


def test_malformed_keys_are_rejected(ctx, circuits):
    _, _, circuit = circuits["chain8"]
    raw = bytes(circuit.verifying_key().to_bytes())
    n = circuit.rows
    off = ref.layout(n)

    def put(at, data, base=raw):
        b = bytearray(base)
        b[at:at + len(data)] = data
        return b

    for check in (0, 1, 2):
        _expect_malformed(ctx, raw[:-1], check, ["length"])
        _expect_malformed(ctx, raw + b"\0", check, ["length"])
        _expect_malformed(ctx, raw[:100], check, ["truncated"])
        _expect_malformed(ctx, put(0, b"TPVX"), check, ["tag"])
        _expect_malformed(ctx, put(4, (2).to_bytes(4, "little")), check, ["version"])
        _expect_malformed(ctx, put(8, (n + 1).to_bytes(8, "little")), check, ["power of two"])
        _expect_malformed(ctx, put(off["sigma_1_len"], (n - 1).to_bytes(8, "little")), check, ["sigma_1 length"])
        _expect_malformed(ctx, put(off["sigma_2_len"], (n + 1).to_bytes(8, "little")), check, ["sigma_2 length"])
        for idx in (0, n // 2, n - 1):
            _expect_malformed(ctx, put(off["sigma_1"] + 32 * idx, R_MOD.to_bytes(32, "little")), check, ["sigma_1[%d]" % idx])
        _expect_malformed(ctx, put(off["sigma_2"] + 32 * (n - 1), (R_MOD + 5).to_bytes(32, "little")), check, ["sigma_2[%d]" % (n - 1)])
        _expect_malformed(ctx, put(off["k"] + 32, R_MOD.to_bytes(32, "little")), check, ["k[1]"])
        _expect_malformed(ctx, put(off["g1"] + 96 * 2, Q_MOD.to_bytes(48, "little")), check, ["q_o"])
        g2s_bad = bytearray(raw[off["g2s"]: off["sigma_1_len"]])
        g2s_bad[100] ^= 1
        _expect_malformed(ctx, put(off["g2s"], g2s_bad), check, ["g2s"])
    # a point off the curve: rejected from check 1 on
    off_curve = put(off["g1"] + 96 * 0, (1).to_bytes(48, "little") + (1).to_bytes(48, "little"))
    VerifyingKey.from_bytes(ctx, bytes(off_curve), 0)
    for check in (1, 2):
        _expect_malformed(ctx, off_curve, check, ["q_l"])
    # the order-3 point (0, 2) as the sigma_3 commitment: on the curve, outside the prime-order subgroup
    order3 = put(off["g1"] + 96 * 7, (0).to_bytes(48, "little") + (2).to_bytes(48, "little"))
    VerifyingKey.from_bytes(ctx, bytes(order3), 0)
    VerifyingKey.from_bytes(ctx, bytes(order3), 1)
    _expect_malformed(ctx, order3, 2, ["sigma_3 commitment", "subgroup"])


def _pairs(circuits, names, per_key, seed=0):
    keys = {name: circuits[name][2].verifying_key() for name in names}
    lists = {name: proofs_of(circuits[name][2], per_key, seed) for name in names}
    pairs = []
    for k in range(per_key):   # interleaved
        for name in names:
            pairs.append((keys[name], lists[name][k]))
    return keys, pairs


def test_batch_over_several_keys(ctx, circuits):
    names = ["readme", "additive", "chain10", "chain12"]
    keys, pairs = _pairs(circuits, names, 16)
    assert len(pairs) == 64
    all_ok, each = verify_batch(pairs)
    assert all_ok and each == [True] * 64
    # one corrupted proof per key: localised, and each verdict equals VerifyingKey.verify
    bad = list(pairs)
    for j, name in enumerate(names):
        at = 4 * (3 + 2 * j) + j
        assert bad[at][0] is keys[name]
        bad[at] = (keys[name], corrupt(bad[at][1], CORRUPTIONS[2 + j]))
    all_ok, each = verify_batch(bad)
    assert not all_ok
    singles = [outcome(vk.verify, p) is True for vk, p in bad]
    assert each == singles and singles.count(False) == 4
    # a proof attributed to another key is rejected, the rest accepted
    swapped = list(pairs)
    swapped[5] = (keys["chain12"], pairs[5][1])
    all_ok, each = verify_batch(swapped)
    assert not all_ok and each == [k != 5 for k in range(64)]


def test_batch_over_two_srs_groups(ctx):
    desc = mul_chain(253)
    a, b = desc.build(ctx, TAU), desc.build(ctx, TAU2)
    ka, kb = a.verifying_key(), b.verifying_key()
    pa, pb = proofs_of(a, 6), proofs_of(b, 6, seed=50)
    pairs = [(ka, p) for p in pa] + [(kb, p) for p in pb]
    assert verify_batch(pairs) == (True, [True] * 12)
    crossed = list(pairs)
    crossed[2] = (kb, pa[2])
    crossed[9] = (ka, pb[3])
    all_ok, each = verify_batch(crossed)
    assert not all_ok and each == [k not in (2, 9) for k in range(12)]


def test_one_key_agrees_with_circuit_batch(ctx, circuits):
    _, _, circuit = circuits["chain8"]
    vk = circuit.verifying_key()
    proofs = proofs_of(circuit, 24, seed=100)
    for j in (3, 17):
        proofs[j] = corrupt(proofs[j], 224 + 192)
    proofs[20] = Proof(proofs[20].fixed, [9] + [0] * (circuit.rows - 1))
    assert verify_batch([(vk, p) for p in proofs]) == circuit.verify_batch(proofs)
    assert verify_batch([]) == (True, [])


def test_argument_errors(ctx, circuits):
    _, _, circuit = circuits["readme"]
    vk = circuit.verifying_key()
    p = proofs_of(circuit, 1)[0]
    other = Context(0)
    try:
        foreign = mul_chain(13).build(other, TAU).verifying_key()
        with pytest.raises(TyplonkError):
            verify_batch([(vk, p), (foreign, p)])
        with pytest.raises(TyplonkError):
            ctx.vk_verify_batch([vk.handle], [1], [p.fixed], [b""])        # key index out of range
        with pytest.raises(TyplonkError):
            ctx.vk_verify_batch([vk.handle], [0], [p.fixed], [bytes(32 * (circuit.rows + 1))])   # more inputs than rows
        with pytest.raises(TyplonkError):
            ctx.vk_verify_batch([vk.handle], [0], [p.fixed], [R_MOD.to_bytes(32, "little")])    # not reduced
        with pytest.raises(TyplonkError):
            ctx.vk_verify_batch([], [], [], [])                              # no key
        foreign.handle.destroy()
    finally:
        other.close()


def test_device_group_gives_the_same_bytes_and_verdicts(ctx, circuits):
    group = Context.multi([0, 0])
    try:
        names = ["readme", "chain8"]
        gkeys = {}
        for name in names:
            run, n_in, single = circuits[name]
            gc = single.desc.build(group, TAU)
            gkeys[name] = gc.verifying_key()
            raw = gkeys[name].to_bytes()
            assert raw == single.verifying_key().to_bytes()
            assert VerifyingKey.from_bytes(group, raw, 2).to_bytes() == raw
        pairs = []
        for name in names:
            ps = proofs_of(circuits[name][2], 5)
            pairs += [(gkeys[name], p) for p in ps]
        pairs[3] = (pairs[3][0], corrupt(pairs[3][1], 192))
        all_ok, each = verify_batch(pairs)
        assert not all_ok and each == [k != 3 for k in range(10)]
        assert [gkeys[names[k // 5]].verify(p) for k, (_, p) in enumerate(pairs)] == each
        for vk in gkeys.values():
            vk.handle.destroy()
    finally:
        group.close()


def test_at_2_16(ctx):
    circuit = mul_chain((1 << 16) - 3).build(ctx, TAU)
    vk = circuit.verifying_key()
    raw = vk.to_bytes()
    assert len(raw) == 1376 + 64 * (1 << 16)
    back = VerifyingKey.from_bytes(ctx, raw, 2)
    assert back.to_bytes() == raw
    proofs = proofs_of(circuit, 16)
    proofs[7] = corrupt(proofs[7], 1024 + 1)
    all_ok, each = verify_batch([(back, p) for p in proofs])
    assert not all_ok and each == [k != 7 for k in range(16)]


def test_cpp_mirror(tmp_path):
    from typlonk_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "typlonk_b200", "lib")
    exe = str(tmp_path / "verify_key_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                          "-o", exe, os.path.join(ROOT, "tests", "cpp", "verify_key_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout, res.stdout + res.stderr
    assert "0 failures" in res.stdout
