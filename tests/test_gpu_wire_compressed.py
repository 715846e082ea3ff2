"""GPU tests of the compressed wire encodings (csrc/wire.cu): the SRS codec, whose square roots and checks run on the
device, against the reference codec (wire_compressed_ref.py) and the uncompressed codec; batch decompression of proofs
(tp_proofs_decompress) against the host decoder; device groups; the C++ mirror."""
import os
import struct
import subprocess

import pytest

import wire_compressed_ref as ref
from oracle.pyoracle import curve, fields, kzg as okzg, rng
from typlonk_b200 import field as F, ffi, synthetic
from typlonk_b200.ffi import Context, PROOF_COMPRESSED_FIXED_BYTES, PROOF_FIXED_BYTES
from typlonk_b200.kzg import KzgScheme, Srs

from test_gpu_prove import TAU, mul_chain

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = fields.Q_MOD, fields.R_MOD


def _no_root_x():
    x = 1
    while pow((x ** 3 + 4) % Q, (Q - 1) // 2, Q) == 1:
        x += 1
    return x


def _off_subgroup_point():
    """a curve point outside the prime-order subgroup: [r - 1]P != -P (the oracle's g1_mul reduces mod r)"""
    x = 0
    while True:
        x += 1
        rhs = (x ** 3 + 4) % Q
        y = pow(rhs, (Q + 1) // 4, Q)
        if y * y % Q == rhs and curve.g1_mul((x, y), R - 1) != curve.g1_neg((x, y)):
            return (x, y)


def test_srs_compressed_bytes_equal_the_reference_and_round_trip(ctx):
    gates = 29
    srs = Srs.from_secret(ctx, TAU, gates)
    raw = srs.to_bytes(compressed=True)
    osrs = okzg.Srs.from_secret(TAU, gates)
    want = struct.pack("<Q", gates + 3) + b"".join(ref.g1_serialize_compressed(p) for p in osrs.g1)
    want += ref.g2_serialize_compressed(osrs.g2) + ref.g2_serialize_compressed(osrs.g2s)
    assert raw == want
    assert len(raw) == 8 + 48 * (gates + 3) + 192
    poly = rng.fr_rand_stream(9, gates + 3)
    for check in (0, 1, 2):
        back = Srs.from_bytes(ctx, raw, check, compressed=True)
        assert back.handle.download() == srs.handle.download()
        assert back.handle.g2() == srs.handle.g2()
        assert KzgScheme(back).commit(poly) == KzgScheme(srs).commit(poly)
        assert back.to_bytes() == srs.to_bytes()
        assert back.to_bytes(compressed=True) == raw


def test_srs_compressed_at_scale_subgroup_checked(ctx):
    """2^16 + 3 points: compressed serialisation, device decompression with the full subgroup check."""
    srs = Srs.from_secret(ctx, TAU, 1 << 16)
    raw = srs.to_bytes(compressed=True)
    assert len(raw) == 8 + 48 * ((1 << 16) + 3) + 192
    back = Srs.from_bytes(ctx, raw, 2, compressed=True)
    assert back.handle.download() == srs.handle.download()
    assert back.to_bytes() == srs.to_bytes()


def test_golden_2_16_proof_from_a_compressed_srs(ctx):
    import json
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "mulchain_big.json")))["2^16"]["proof_hex"]
    n = 1 << 16
    first = Srs.from_secret(ctx, synthetic.tau(), n)
    raw = first.to_bytes(compressed=True)
    first.handle.destroy()
    srs = Srs.from_bytes(ctx, raw, 2, compressed=True)
    t = synthetic.mul_chain_trace(n - 3)
    sel_all = t.selectors()
    sel = [bytes(sel_all[k * n * 32:(k + 1) * n * 32]) for k in range(5)]
    handle, _ = ctx.circuit_compile(srs.handle, sel, bytes(t.permutation()), n)
    cols = [F.fr_vec_to_bytes(c) for c in synthetic.mul_chain_witness(n - 3, n)]
    assert handle.prove_inputs(cols, bytes(32)).hex() == gold
    handle.destroy()
    srs.handle.destroy()


def test_srs_compressed_rejections(ctx):
    raw = bytearray(Srs.from_secret(ctx, TAU, 61).to_bytes(compressed=True))
    n = 64

    def at(i):
        return 8 + 48 * i

    def expect(bad, check, index=None):
        with pytest.raises(ffi.Malformed) as e:
            Srs.from_bytes(ctx, bytes(bad), check, compressed=True)
        if index is not None:
            assert "first at index %d" % index in str(e.value), str(e.value)

    for cut in (raw[:-1], raw + b"\0", raw[:8 + 191]):
        with pytest.raises(ffi.Malformed):
            Srs.from_bytes(ctx, bytes(cut), 0, compressed=True)
    bad = bytearray(raw)
    bad[0:8] = struct.pack("<Q", n + 1)
    expect(bad, 0)
    # x >= q
    bad = bytearray(raw)
    bad[at(17):at(18)] = Q.to_bytes(48, "little")
    expect(bad, 0, 17)
    # an x without a root: rejected at every check level
    bad = bytearray(raw)
    bad[at(23):at(24)] = _no_root_x().to_bytes(48, "little")
    for check in (0, 1, 2):
        expect(bad, check, 23)
    # both flags; infinity with x != 0; infinity with the sign bit
    for i, mutate in ((30, lambda r: r.__setitem__(47, r[47] | 0xC0)),
                      (31, lambda r: r.__setitem__(47, (r[47] & 0x3F) | 0x40)),
                      (32, lambda r: r.__setitem__(slice(0, 48), bytes(47) + b"\xc0"))):
        bad = bytearray(raw)
        rec = bytearray(bad[at(i):at(i + 1)])
        mutate(rec)
        bad[at(i):at(i + 1)] = rec
        expect(bad, 0, i)
    # off the subgroup: accepted at check 1, rejected at check 2 -- a generic point and the order-3 point (0, 2)
    for i, pt in ((40, _off_subgroup_point()), (41, (0, 2)), (42, (0, Q - 2))):
        bad = bytearray(raw)
        bad[at(i):at(i + 1)] = ref.g1_serialize_compressed(pt)
        s = Srs.from_bytes(ctx, bytes(bad), 1, compressed=True)
        assert F.g1_from_packed(s.handle.download(i, 1)) == pt
        s.handle.destroy()
        expect(bad, 2, i)
    # two bad records: the lowest index is reported
    bad = bytearray(raw)
    bad[at(40):at(41)] = ref.g1_serialize_compressed((0, 2))
    bad[at(5):at(6)] = Q.to_bytes(48, "little")
    expect(bad, 2, 5)
    # a malformed G2 point: both flags, and an x without a root in Fq2 (found by search)
    tail = 8 + 48 * n
    bad = bytearray(raw)
    bad[tail + 95] |= 0xC0
    expect(bad, 0)
    x0 = 1
    while True:
        try:
            ref.g2_deserialize_compressed(x0.to_bytes(48, "little") + bytes(48))
        except ValueError:
            break
        x0 += 1
    bad = bytearray(raw)
    bad[tail + 96:tail + 192] = x0.to_bytes(48, "little") + bytes(48)
    expect(bad, 0)


def test_infinity_record_round_trips(ctx):
    raw = bytearray(Srs.from_secret(ctx, TAU, 29).to_bytes(compressed=True))
    raw[8 + 48 * 7:8 + 48 * 8] = ref.g1_serialize_compressed(None)
    s = Srs.from_bytes(ctx, bytes(raw), 2, compressed=True)
    assert s.handle.download(7, 1) == bytes(96)
    assert bytes(s.to_bytes(compressed=True)) == bytes(raw)


def _corrupt(block: bytes, k: int) -> bytes:
    """a few kinds of damage to a compressed proof block, chosen by k"""
    b = bytearray(block)
    kind = k % 6
    if kind == 0:
        b[47] |= 0xC0                                    # a.commitment: both flags
    elif kind == 1:
        b[48:96] = Q.to_bytes(48, "little")             # a.W: x = q
    elif kind == 2:
        b[0:48] = _no_root_x().to_bytes(48, "little")   # no root
    elif kind == 3:
        b[96:128] = R.to_bytes(32, "little")            # a.y = r
    elif kind == 4:
        b[47] ^= 0x80                                    # a sign flip: still a valid block
    else:
        b[0:48] = ref.g1_serialize_compressed((0, 2))    # order 3: decodes (no subgroup check here)
    return bytes(b)


def _batch_vs_host(ctx, blocks):
    count = len(blocks)
    got, status = ctx.proofs_decompress(b"".join(blocks), count)
    for k, blk in enumerate(blocks):
        try:
            want, st = ffi.proof_decompress(blk), 0
        except ffi.Malformed:
            want, st = bytes(PROOF_FIXED_BYTES), 12
        assert status[k] == st, k
        assert got[k * PROOF_FIXED_BYTES:(k + 1) * PROOF_FIXED_BYTES] == want, k
    return got, status


def test_proofs_decompress_matches_the_host_decoder(ctx):
    import json
    proofs = json.load(open(os.path.join(ROOT, "tests", "golden", "proofs.json")))
    good = [ffi.proof_compress(bytes.fromhex(p["proof_hex"])[:PROOF_FIXED_BYTES]) for p in proofs.values()]
    blocks = []
    for k in range(1000):
        g = good[k % len(good)]
        blocks.append(_corrupt(g, k // 2) if k % 2 else g)
    got, status = _batch_vs_host(ctx, blocks)
    assert 0 < status.count(12) < 1000
    # status == NULL: the lowest failing index is returned and named
    first = status.index(12)
    out = (ffi.C.c_char * (1000 * PROOF_FIXED_BYTES))()
    rc = ffi.lib().tp_proofs_decompress(ctx._h, ffi._buf(b"".join(blocks)), ffi.C.c_size_t(1000), out,
                                        ffi.C.c_size_t(1000 * PROOF_FIXED_BYTES), None)
    assert rc == 12
    assert "proof %d " % first in ffi.lib().tp_last_error(ctx._h).decode()
    assert bytes(out) == got
    # argument errors
    with pytest.raises(ffi.TyplonkError) as e:
        ctx.proofs_decompress(b"".join(good[:1]) * 65537, 65537)
    assert e.value.code == 1
    rc = ffi.lib().tp_proofs_decompress(ctx._h, ffi._buf(good[0]), ffi.C.c_size_t(1), out, ffi.C.c_size_t(100), None)
    assert rc == 9
    assert ctx.proofs_decompress(b"", 0) == (b"", [])


def test_prove_batch_compress_decompress_verify_batch(ctx):
    circuit = mul_chain(13).build(ctx, TAU)
    count = 12
    ins = [[3 + k, 5 + k] for k in range(count)]
    bls = [rng.fr_rand_stream(7000 + k, 9) for k in range(count)]
    proofs = circuit.prove_batch(ins, [[0]] * count, bls)
    blob = b"".join(ffi.proof_compress(p.fixed) for p in proofs)
    assert len(blob) == count * PROOF_COMPRESSED_FIXED_BYTES
    fixed, status = ctx.proofs_decompress(blob, count)
    assert status == [0] * count
    assert [fixed[k * PROOF_FIXED_BYTES:(k + 1) * PROOF_FIXED_BYTES] for k in range(count)] == [p.fixed for p in proofs]
    all_ok, each = circuit.handle.verify_batch(
        [fixed[k * PROOF_FIXED_BYTES:(k + 1) * PROOF_FIXED_BYTES] for k in range(count)],
        [F.fr_vec_to_bytes(p.public_inputs) for p in proofs])
    assert all_ok and all(each)
    # the Proof surface round-trips through the compressed framing
    from typlonk_b200.plonk import Proof
    enc = proofs[0].to_bytes(compressed=True)
    assert len(enc) == 848 + 8 + 32 * circuit.rows
    assert circuit.verify(Proof.from_bytes(enc, compressed=True))


def test_device_group_of_two_ranks_on_one_device():
    g = Context.multi([0, 0])
    try:
        srs = Srs.from_secret(g, TAU, 61)
        raw = srs.to_bytes(compressed=True)
        single = Context(0)
        try:
            assert raw == Srs.from_secret(single, TAU, 61).to_bytes(compressed=True)
            back = Srs.from_bytes(g, raw, 2, compressed=True)
            assert len(back) == 64
            assert back.to_bytes() == srs.to_bytes()
            poly = rng.fr_rand_stream(9, 64)
            assert KzgScheme(back).commit(poly) == KzgScheme(srs).commit(poly)
            bad = bytearray(raw)
            bad[8 + 48 * 9:8 + 48 * 10] = ref.g1_serialize_compressed((0, 2))
            with pytest.raises(ffi.Malformed) as e:
                Srs.from_bytes(g, bytes(bad), 2, compressed=True)
            assert "first at index 9" in str(e.value)
            import json
            proofs = json.load(open(os.path.join(ROOT, "tests", "golden", "proofs.json")))
            good = [ffi.proof_compress(bytes.fromhex(p["proof_hex"])[:PROOF_FIXED_BYTES]) for p in proofs.values()]
            blocks = [(_corrupt(b, k) if k % 3 == 1 else b) for k, b in enumerate(good * 4)]
            want = single.proofs_decompress(b"".join(blocks), len(blocks))
            assert g.proofs_decompress(b"".join(blocks), len(blocks)) == want
            _batch_vs_host(g, blocks)
        finally:
            single.close()
    finally:
        g.close()


def test_cpp_wire_compressed(tmp_path):
    from typlonk_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "typlonk_b200", "lib")
    exe = str(tmp_path / "wire_compressed_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                          "-o", exe, os.path.join(ROOT, "tests", "cpp", "wire_compressed_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout and "0 failures" in res.stdout, res.stdout + res.stderr
