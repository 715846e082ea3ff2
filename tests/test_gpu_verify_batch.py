"""GPU tests of batch verification (tp_verify_batch through CircuitHandle.verify_batch / CompiledCircuit.verify_batch):
honest batches of every size class, localisation of bad proofs among good ones with the same verdicts as tp_verify,
the subgroup check, argument errors, device groups, proofs at 2^16 and 2^20 and the C++ mirror."""
import ctypes as C
import os
import subprocess

import pytest

from oracle.pyoracle import curve, fields
from typlonk_b200 import field as F, synthetic
from typlonk_b200.ffi import Context, PROOF_FIXED_BYTES, TyplonkError, lib
from typlonk_b200.plonk import Proof

from test_gpu_prove import Additive, Pythagoras, mul_chain, BLINDERS, TAU
from test_verify_batch_oracle import cancelling_pair

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORRUPTIONS = (5, 96 + 7, 192, 672 + 3, 1024 + 1, 1056 + 9, 1344 + 2, 1440)   # test_mul_chain_verify_and_corruption


def blinders(seed):
    from oracle.pyoracle import rng
    return rng.fr_rand_stream(1000 + seed, 9)


def honest(circuit, count, inputs):
    return [circuit.prove(inputs(k), [0], blinders(k)) for k in range(count)]


def expect_verdicts(circuit, proofs, expected=None):
    singles = [circuit.verify(p) for p in proofs]
    if expected is not None:
        assert singles == expected
    all_ok, each = circuit.verify_batch(proofs)
    assert each == singles
    assert all_ok == all(singles)
    return each


@pytest.fixture(scope="module")
def chain(ctx):
    circuit = mul_chain(253).build(ctx, TAU)
    return circuit, honest(circuit, 64, lambda k: [3 + k, 5 + 2 * k])


@pytest.mark.parametrize("count", [1, 2, 7, 64])
def test_honest_batches_mul_chain(chain, count):
    circuit, proofs = chain
    assert expect_verdicts(circuit, proofs[:count], [True] * count) == [True] * count


@pytest.mark.parametrize("count", [1, 2, 7, 64])
def test_honest_batches_additive(ctx, count):
    circuit = Additive.build(ctx, TAU)
    # a + b == c + d + e
    proofs = honest(circuit, count, lambda k: [2 + k, 7, 2, 3 + k, 4])
    expect_verdicts(circuit, proofs, [True] * count)


def test_empty_batch(chain):
    circuit, _ = chain
    assert circuit.verify_batch([]) == (True, [])


@pytest.mark.parametrize("off", CORRUPTIONS)
def test_one_corrupted_proof_is_localised(chain, off):
    circuit, proofs = chain
    batch = list(proofs[:16])
    j = 11
    bad = bytearray(batch[j].fixed)
    bad[off] ^= 1
    batch[j] = Proof(bytes(bad), batch[j].public_inputs)
    # a flipped bit can make a coordinate non-canonical: tp_verify then raises, the batch only rejects
    try:
        expected_single = circuit.verify(batch[j])
    except TyplonkError:
        expected_single = False
    assert not expected_single
    all_ok, each = circuit.verify_batch(batch)
    assert not all_ok and each == [k != j for k in range(16)]


def test_mixed_bad_proofs(ctx, chain):
    circuit, proofs = chain
    batch = list(proofs[:16])
    for j in (3, 12):   # two bad proofs
        bad = bytearray(batch[j].fixed)
        bad[224 + 192] ^= 1
        batch[j] = Proof(bytes(bad), batch[j].public_inputs)
    other = mul_chain(13).build(ctx, TAU).prove([3, 5], [0], BLINDERS)
    batch[5] = Proof(other.fixed, batch[5].public_inputs)                     # a proof of a different circuit
    batch[7] = Proof(batch[7].fixed, [1])                                    # wrong public inputs
    batch[8] = Proof(batch[8].fixed, [])                                     # short public inputs: resized, accepted
    bad = bytearray(batch[9].fixed)
    bad[96:96 + 96] = F.g1_serialize_unchecked(None)                         # a(zeta)'s witness -> infinity
    batch[9] = Proof(bytes(bad), batch[9].public_inputs)
    expected = [k not in (3, 12, 5, 7, 9) for k in range(16)]
    expect_verdicts(circuit, batch, expected)
    bad = bytearray(batch[10].fixed)
    bad[0:48] = fields.Q_MOD.to_bytes(48, "little")                          # non-canonical coordinate x = q
    batch[10] = Proof(bytes(bad), batch[10].public_inputs)
    with pytest.raises(TyplonkError):
        circuit.verify(batch[10])
    all_ok, each = circuit.verify_batch(batch)
    assert not all_ok and each == [e and k != 10 for k, e in enumerate(expected)]


def test_dishonest_pythagoras_among_honest(ctx):
    circuit = Pythagoras.build(ctx, TAU)
    proofs = [circuit.prove([3, 4, 5], [0], blinders(k)) for k in range(9)]
    proofs[6] = circuit.prove([3, 4, 6], [0], blinders(6))                   # builder/test.rs:31-37
    expect_verdicts(circuit, proofs, [k != 6 for k in range(9)])


def test_cancelling_pair_is_rejected(chain):
    """Two copies of one proof with W_a + D and W_a - D: with all weights 1 the sum would accept."""
    circuit, proofs = chain
    first, second = cancelling_pair(proofs[0].fixed)
    batch = [Proof(first, proofs[0].public_inputs), Proof(second, proofs[0].public_inputs)]
    assert circuit.verify_batch(batch) == (False, [False, False])


def _cofactor_point():
    x = 0
    while True:
        x += 1
        rhs = (x ** 3 + 4) % fields.Q_MOD
        y = pow(rhs, (fields.Q_MOD + 1) // 4, fields.Q_MOD)
        if y * y % fields.Q_MOD == rhs and curve.g1_mul((x, y), fields.R_MOD - 1) != curve.g1_neg((x, y)):
            return x, y


def test_point_outside_the_subgroup_is_rejected(chain):
    circuit, proofs = chain
    x, y = _cofactor_point()
    batch = list(proofs[:4])
    for j, off in ((1, 96), (3, 1056 + 96)):   # a's witness; the second quotient slice (not in the transcript either)
        bad = bytearray(batch[j].fixed)
        bad[off:off + 96] = x.to_bytes(48, "little") + y.to_bytes(48, "little")
        batch[j] = Proof(bytes(bad), batch[j].public_inputs)
    all_ok, each = circuit.verify_batch(batch)
    assert not all_ok and each == [True, False, True, False]


def test_argument_errors(chain):
    circuit, proofs = chain
    h = circuit.handle
    with pytest.raises(TyplonkError):
        h.verify_batch([proofs[0].fixed], [bytes(32 * (circuit.rows + 1))])   # n_public > n
    with pytest.raises(TyplonkError):
        h.verify_batch([proofs[0].fixed], [fields.R_MOD.to_bytes(32, "little")])  # not reduced
    L = lib()
    blob = (C.c_char * PROOF_FIXED_BYTES).from_buffer_copy(proofs[0].fixed)
    zero, one = (C.c_size_t * 1)(0), (C.c_size_t * 1)(1)
    ok = C.c_int(0)
    each = (C.c_int * 1)()
    c, x = h.ctx._h, h._h
    for args in [(x, blob, 1, None, zero, None),          # all_ok null
                 (x, None, 1, None, zero, C.byref(ok)),   # proofs null
                 (x, blob, 1, None, None, C.byref(ok)),   # n_public null
                 (None, blob, 1, None, zero, C.byref(ok)),  # circuit null
                 (x, blob, 1, None, one, C.byref(ok)),    # public-input vectors null with n_public = 1
                 (x, blob, 65537, None, zero, C.byref(ok))]:
        rc = L.tp_verify_batch(c, args[0], args[1], C.c_size_t(args[2]), args[3], args[4], args[5], each)
        assert rc == 1, args


@pytest.mark.parametrize("world", [2, 3])
def test_device_group_same_verdicts(world):
    mctx = Context.multi([0] * world)
    try:
        circuit = mul_chain(253).build(mctx, TAU)
        proofs = honest(circuit, 12, lambda k: [3 + k, 5])
        assert circuit.verify_batch(proofs) == (True, [True] * 12)
        bad = bytearray(proofs[9].fixed)
        bad[192] ^= 1
        proofs[9] = Proof(bytes(bad), proofs[9].public_inputs)
        assert circuit.verify_batch(proofs) == (False, [k != 9 for k in range(12)])
        circuit.handle.destroy()
        circuit.srs.handle.destroy()
    finally:
        mctx.close()


def _large(ctx, log_n, distinct):
    n = 1 << log_n
    circuit = synthetic.mul_chain_direct(ctx, log_n)
    fixed = []
    for k in range(distinct):
        cols = synthetic.mul_chain_witness(n - 3, n, x0=3 + k, blind=blinders(k))
        fixed.append(circuit.handle.prove([F.fr_vec_to_bytes(c) for c in cols], bytes(32 * n)))
    return circuit, fixed


def test_scale_2_16(ctx):
    circuit, fixed = _large(ctx, 16, 3)
    batch = [fixed[0]] * 256 + fixed[1:]
    bad = bytearray(fixed[0])
    bad[224 + 192] ^= 1
    batch[200] = bytes(bad)
    all_ok, each = circuit.handle.verify_batch(batch, [bytes(32)] * len(batch))
    assert not all_ok and each == [k != 200 for k in range(len(batch))]
    assert circuit.handle.verify_batch(batch[:200] + batch[201:], [b""] * (len(batch) - 1)) == (True, [True] * (len(batch) - 1))
    circuit.handle.destroy()
    circuit.srs.handle.destroy()


def test_scale_2_20(ctx):
    circuit, fixed = _large(ctx, 20, 1)
    batch = [fixed[0]] * 64
    bad = bytearray(fixed[0])
    bad[224 + 192] ^= 1
    batch[37] = bytes(bad)
    all_ok, each = circuit.handle.verify_batch(batch, [bytes(32)] * 64)
    assert not all_ok and each == [k != 37 for k in range(64)]
    assert circuit.handle.verify(fixed[0], bytes(32)) and not circuit.handle.verify(bytes(bad), bytes(32))
    circuit.handle.destroy()
    circuit.srs.handle.destroy()


def test_cpp_verify_batch(tmp_path):
    from typlonk_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "typlonk_b200", "lib")
    exe = str(tmp_path / "verify_batch_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                          "-o", exe, os.path.join(ROOT, "tests", "cpp", "verify_batch_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout and "0 failures" in res.stdout, res.stdout + res.stderr
