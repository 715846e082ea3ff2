"""GPU tests of batch proving (tp_prove_batch through CircuitHandle.prove_batch / CompiledCircuit.prove_batch): every
proof of a batch is byte-identical to the single-proof call on the same inputs -- across wave boundaries, for failing
and unusual witnesses, at 2^16..2^20 and on device groups -- the circuit's own buffers are left alone, argument errors
are refused and the C++ mirror agrees."""
import ctypes as C
import json
import os
import subprocess

import pytest

from oracle.pyoracle import builder as obuilder, plonk as oplonk, rng
from typlonk_b200 import field as F, synthetic
from typlonk_b200.ffi import Context, GateUnsatisfied, PROOF_FIXED_BYTES, TyplonkError, lib

import py_tracer
from test_gpu_prove import Additive, Pythagoras, mul_chain, TAU

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WAVE_CAP = 64   # prove_batch.cu


def blinders(seed):
    return rng.fr_rand_stream(5000 + seed, 9)


# Pythagoras checks a^2 + b^2 == c^2 through a copy constraint: a broken triple still proves (a proof that does not
# verify, as the reference makes), so odd k take the floor-quotient path
CASES = {
    "pythagoras": (Pythagoras, lambda k: [3 * (k + 1), 4 * (k + 1), 5 * (k + 1) + (k % 2)]),
    "additive": (Additive, lambda k: [2 + k, 7, 2, 3 + k, 4]),
    **{"mul_chain_%d" % g: (mul_chain(g), lambda k: [3 + k, 5 + 3 * k]) for g in (5, 13, 61, 253)},
}


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("count", [1, 2, 7])
def test_batch_equals_single_proofs(ctx, name, count):
    desc, inputs = CASES[name]
    circuit = desc.build(ctx, TAU)
    ins = [inputs(k) for k in range(count)]
    bls = [blinders(k) for k in range(count)]
    want = [circuit.prove(i, [0], b).fixed for i, b in zip(ins, bls)]
    got = circuit.prove_batch(ins, [[0]] * count, bls)
    assert [p.fixed for p in got] == want
    assert all(p.public_inputs == [0] * circuit.rows for p in got)
    if name in ("pythagoras", "mul_chain_13") and count == 2:
        oc = obuilder.compile_circuit(obuilder.circuit_pythagoras, 3, TAU) if name == "pythagoras" else \
            obuilder.compile_circuit(obuilder.make_mul_chain(13), 2, TAU)
        for i, b, p in zip(ins, bls, got):
            assert oplonk.prove(oc, i, [0], b).to_bytes()[:PROOF_FIXED_BYTES] == p.fixed


def test_wave_boundary(ctx):
    circuit = mul_chain(5).build(ctx, TAU)
    count = WAVE_CAP + 3
    ins = [[3 + k, 5 + k] for k in range(count)]
    bls = [blinders(k) for k in range(count)]
    got = circuit.prove_batch(ins, [[0]] * count, bls)
    assert ctx.get_stat("prove_batch_wave") == WAVE_CAP          # two waves: 64, then 3
    want = [circuit.prove(i, [0], b).fixed for i, b in zip(ins, bls)]
    assert [p.fixed for p in got] == want


def _mixed(circuit):
    """honest, broken copy (floor quotient), compensated non-zero PI (general path), uncompensated non-zero PI."""
    n = circuit.rows
    honest = py_tracer.witness(circuit.desc, n, [3, 4, 5], blinders(1))
    broken = py_tracer.witness(circuit.desc, n, [3, 4, 6], blinders(2))
    base = py_tracer.witness(circuit.desc, n, [5, 12, 13], blinders(3))
    pis = [0] * n
    pis[0] = 9
    cols = lambda w: [F.fr_vec_to_bytes(c) for c in w]  # noqa: E731
    # row 0 is the first gate (a * a, a Mul row): c = a b + PI keeps its gate line at zero
    comp = [list(c) for c in base]
    comp[2][0] = (comp[0][0] * comp[1][0] + pis[0]) % F.R_MOD
    circuit.handle.prove_inputs(cols(comp), F.fr_vec_to_bytes(pis))   # the compensated witness passes the gate check
    return [(cols(honest), b""), (cols(broken), b""), (cols(comp), F.fr_vec_to_bytes(pis)),
            (cols(honest), F.fr_vec_to_bytes(pis))]


def _singles(handle, items):
    out = []
    for cols, pi in items:
        try:
            out.append((handle.prove_inputs(cols, pi), 0))
        except TyplonkError as e:
            out.append((bytes(PROOF_FIXED_BYTES), e.code))
    return out


def _check_mixed(handle, items):
    want = _singles(handle, items)
    assert [s for _, s in want] == [0, 0, 0, 6]
    for order in (list(range(4)), [3, 2, 1, 0]):
        batch = [items[i] for i in order]
        fixed, status = handle.prove_batch([c for c, _ in batch], [p for _, p in batch])
        assert status == [want[i][1] for i in order]
        assert fixed == [want[i][0] for i in order]
    return want


def test_mixed_batch(ctx):
    circuit = Pythagoras.build(ctx, TAU)
    items = _mixed(circuit)
    _check_mixed(circuit.handle, items)
    # status NULL: the first failure's code, its index named
    L = lib()
    count = len(items)
    keep = [(C.c_char * len(b)).from_buffer_copy(b) for cols, _ in items for b in cols]
    adv = (C.c_void_p * (3 * count))(*[C.cast(b, C.c_void_p) for b in keep])
    pk = [(C.c_char * len(p)).from_buffer_copy(p) if p else None for _, p in items]
    pis = (C.c_void_p * count)(*[C.cast(b, C.c_void_p) if b is not None else None for b in pk])
    npub = (C.c_size_t * count)(*[len(p) // 32 for _, p in items])
    out = (C.c_char * (count * PROOF_FIXED_BYTES))()
    rc = L.tp_prove_batch(ctx._h, circuit.handle._h, C.c_size_t(count), adv, pis, npub, out,
                          C.c_size_t(count * PROOF_FIXED_BYTES), None)
    assert rc == 6 and "proof 3" in L.tp_last_error(ctx._h).decode()
    with pytest.raises(GateUnsatisfied, match="proof 1"):
        circuit.prove_batch([[3, 4, 5], [3, 4, 5]], [[0], [1]], [blinders(0), blinders(1)])


@pytest.mark.parametrize("log_n,count", [(16, 3), (18, 3), (20, 2)])
def test_goldens(ctx, log_n, count):
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "mulchain_big.json")))["2^%d" % log_n]
    n = 1 << log_n
    circuit = synthetic.mul_chain_direct(ctx, log_n)
    cols = [F.fr_vec_to_bytes(c) for c in synthetic.mul_chain_witness(n - 3, n)]
    fixed, status = circuit.handle.prove_batch([cols] * count, [bytes(32)] * count)
    assert status == [0] * count
    assert all(f.hex() == gold["proof_hex"] for f in fixed)
    circuit.handle.destroy()
    circuit.srs.handle.destroy()


def test_batch_leaves_the_circuit_buffers_alone(ctx):
    circuit = mul_chain(13).build(ctx, TAU)
    h = circuit.handle
    n = circuit.rows
    cols = [F.fr_vec_to_bytes(c) for c in py_tracer.witness(circuit.desc, n, [3, 5], blinders(0))]
    zero = h.prove_inputs(cols, b"")
    polys = [h.read_poly(w) for w in range(7)]
    items = [[F.fr_vec_to_bytes(c) for c in py_tracer.witness(circuit.desc, n, [4 + k, 7], blinders(k))] for k in range(5)]
    pis = [b"", F.fr_vec_to_bytes([0, 0, 7] + [0] * (n - 3)), b"", b"", b""]
    h.prove_batch(items, pis)
    assert [h.read_poly(w) for w in range(7)] == polys
    # the zero-PI fast path of the circuit (pi_buffers_zero) must still be right, alternating with non-zero PI
    nz_pis = [0] * n
    nz_pis[2] = 7
    nz_cols = [list(c) for c in py_tracer.witness(circuit.desc, n, [3, 5], blinders(0))]
    nz_cols[2][2] = (nz_cols[0][2] * nz_cols[1][2] + 7) % F.R_MOD
    nz_cols = [F.fr_vec_to_bytes(c) for c in nz_cols]
    nz = h.prove_inputs(nz_cols, F.fr_vec_to_bytes(nz_pis))
    h.prove_batch(items, pis)
    assert h.prove_inputs(cols, b"") == zero
    h.prove_batch(items, pis)
    assert h.prove_inputs(nz_cols, F.fr_vec_to_bytes(nz_pis)) == nz
    h.prove_batch(items, pis)
    assert h.prove_inputs(cols, b"") == zero


def test_argument_errors(ctx):
    circuit = mul_chain(5).build(ctx, TAU)
    h = circuit.handle
    n = circuit.rows
    L = lib()
    col = (C.c_char * (32 * n))()
    adv = (C.c_void_p * 3)(*[C.cast(col, C.c_void_p)] * 3)
    adv_null = (C.c_void_p * 3)(C.cast(col, C.c_void_p), None, C.cast(col, C.c_void_p))
    zero, big = (C.c_size_t * 1)(0), (C.c_size_t * 1)(n + 1)
    out = (C.c_char * PROOF_FIXED_BYTES)(*([7] * PROOF_FIXED_BYTES))
    st = (C.c_int * 1)()
    c, x = ctx._h, h._h
    assert L.tp_prove_batch(c, x, C.c_size_t(0), None, None, None, out, C.c_size_t(0), None) == 0
    assert bytes(out) == bytes([7] * PROOF_FIXED_BYTES)                        # nothing written
    assert L.tp_prove_batch(c, x, C.c_size_t(1), adv_null, None, zero, out, C.c_size_t(PROOF_FIXED_BYTES), st) == 1
    assert L.tp_prove_batch(c, x, C.c_size_t(1), adv, None, big, out, C.c_size_t(PROOF_FIXED_BYTES), st) == 1
    assert L.tp_prove_batch(c, x, C.c_size_t(1), adv, None, zero, out, C.c_size_t(PROOF_FIXED_BYTES - 1), st) == 9
    assert L.tp_prove_batch(c, x, C.c_size_t(65537), adv, None, zero, out, C.c_size_t(PROOF_FIXED_BYTES), st) == 1
    assert L.tp_prove_batch(c, None, C.c_size_t(1), adv, None, zero, out, C.c_size_t(PROOF_FIXED_BYTES), st) == 1


@pytest.mark.parametrize("world", [2, 3])
def test_device_group_same_bytes(ctx, world):
    single = mul_chain(61).build(ctx, TAU)
    ins = [[3 + k, 5 + k] for k in range(7)]
    bls = [blinders(k) for k in range(7)]
    want = [p.fixed for p in single.prove_batch(ins, [[0]] * 7, bls)]
    spy = Pythagoras.build(ctx, TAU)
    items = _mixed(spy)
    want_mixed = spy.handle.prove_batch([c for c, _ in items], [p for _, p in items])
    mctx = Context.multi([0] * world)
    try:
        circuit = mul_chain(61).build(mctx, TAU)
        assert [p.fixed for p in circuit.prove_batch(ins, [[0]] * 7, bls)] == want
        gp = Pythagoras.build(mctx, TAU)
        assert gp.handle.prove_batch([c for c, _ in items], [p for _, p in items]) == want_mixed
        for cc in (circuit, gp):
            cc.handle.destroy()
            cc.srs.handle.destroy()
    finally:
        mctx.close()


def test_batch_proofs_verify(ctx):
    circuit = mul_chain(253).build(ctx, TAU)
    proofs = circuit.prove_batch([[3 + k, 5] for k in range(9)], [[0]] * 9, [blinders(k) for k in range(9)])
    assert circuit.verify_batch(proofs) == (True, [True] * 9)
    assert all(circuit.verify(p) for p in proofs)


def test_cpp_prove_batch(tmp_path):
    from typlonk_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "typlonk_b200", "lib")
    exe = str(tmp_path / "prove_batch_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                          "-o", exe, os.path.join(ROOT, "tests", "cpp", "prove_batch_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout and "0 failures" in res.stdout, res.stdout + res.stderr
