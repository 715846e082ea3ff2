"""Compressed wire encodings (csrc/wire.cu), host side: the reference codec (wire_compressed_ref.py) against itself and
the oracle, and the library's proof codec (tp_proof_compress / decompress / encode_compressed / decode_compressed)
against the reference on every golden proof, with every kind of malformed input."""
import json
import os
import random
import struct

import pytest

import wire_compressed_ref as ref
from oracle.pyoracle import curve, fields, kzg as okzg, rng
from typlonk_b200 import ffi
from typlonk_b200.plonk import Proof

GOLD = os.path.join(os.path.dirname(__file__), "golden")
PROOFS = json.load(open(os.path.join(GOLD, "proofs.json")))
Q, R = fields.Q_MOD, fields.R_MOD


def _golden_fixed(name="readme_pythagoras_3_4_5"):
    return bytes.fromhex(PROOFS[name]["proof_hex"])[:1472]


def _no_root_x():
    """the smallest x >= 1 with x^3 + 4 not a square mod q: no curve point has it"""
    x = 1
    while pow((x ** 3 + 4) % Q, (Q - 1) // 2, Q) == 1:
        x += 1
    return x


def test_reference_round_trips_over_an_oracle_srs():
    srs = okzg.Srs.from_secret(rng.fr_rand_stream(1, 1)[0], 29)
    for p in srs.g1 + [None, curve.g1_neg(srs.g1[3])]:
        b = ref.g1_serialize_compressed(p)
        assert len(b) == 48
        assert ref.g1_deserialize_compressed(b) == p
    for p in (srs.g2, srs.g2s, None, curve.g2_neg(srs.g2)):
        b = ref.g2_serialize_compressed(p)
        assert len(b) == 96
        got = ref.g2_deserialize_compressed(b)
        assert (got is None and p is None) or (got[0] == p[0] and got[1] == p[1])
    # a point and its negation differ exactly in the sign bit
    a, b = ref.g1_serialize_compressed(srs.g1[5]), ref.g1_serialize_compressed(curve.g1_neg(srs.g1[5]))
    assert a[:47] == b[:47] and (a[47] ^ b[47]) == 0x80


def test_sign_bits_of_the_generator_and_17g():
    """G's y (Appendix B) is below (q - 1) / 2, 17 G's is above it."""
    g = curve.G1_GEN
    g17 = curve.g1_mul(g, 17)
    assert g[1] < (Q - 1) // 2 and g17[1] > (Q - 1) // 2
    assert ref.g1_serialize_compressed(g)[47] & 0x80 == 0
    assert ref.g1_serialize_compressed(g17)[47] & 0x80 == 0x80
    assert ref.g1_serialize_compressed(curve.g1_neg(g17))[47] & 0x80 == 0


@pytest.mark.parametrize("name", sorted(PROOFS))
def test_proof_codec_against_the_reference(name):
    raw = bytes.fromhex(PROOFS[name]["proof_hex"])
    fixed = raw[:1472]
    want = ref.proof_block_compress(fixed)
    assert len(want) == ffi.PROOF_COMPRESSED_FIXED_BYTES == 848
    assert ffi.proof_compress(fixed) == want
    assert ffi.proof_decompress(want) == fixed
    enc = ffi.proof_encode_compressed(*ffi.proof_decode(raw))
    assert enc == want + raw[1472:]
    assert ffi.proof_decode_compressed(enc) == ffi.proof_decode(raw)
    p = Proof.from_bytes(enc, compressed=True)
    assert p == Proof.from_bytes(raw)
    assert p.to_bytes(compressed=True) == enc and p.to_bytes() == raw


def test_proof_compress_rejects_what_decode_rejects():
    fixed = bytearray(_golden_fixed())
    for bad_len in (0, 1471, 1473):
        with pytest.raises(ffi.Malformed):
            ffi.proof_compress(bytes(fixed[:bad_len]) if bad_len <= 1472 else bytes(fixed) + b"\0")
    for mutate in (lambda b: b.__setitem__(0, b[0] ^ 1),                          # off the curve
                   lambda b: b.__setitem__(95, b[95] | 0x80),                     # compressed flag in an uncompressed record
                   lambda b: b.__setitem__(slice(192, 224), R.to_bytes(32, "little"))):  # scalar = r
        bad = bytearray(fixed)
        mutate(bad)
        with pytest.raises(ffi.Malformed):
            ffi.proof_decode(bytes(bad) + bytes(8))
        with pytest.raises(ffi.Malformed):
            ffi.proof_compress(bytes(bad))


def _expect_malformed(block):
    with pytest.raises(ffi.Malformed):
        ffi.proof_decompress(bytes(block))
    with pytest.raises(ffi.Malformed):
        ffi.proof_decode_compressed(bytes(block) + bytes(8))


def test_proof_decompress_rejections():
    good = bytearray(ffi.proof_compress(_golden_fixed()))
    # length: truncated block, trailing byte; and the framing
    for blk in (good[:847], good + b"\0"):
        with pytest.raises(ffi.Malformed):
            ffi.proof_decompress(bytes(blk))
    enc = ffi.proof_encode_compressed(_golden_fixed(), b"")
    for cut in (0, 848, len(enc) - 1):
        with pytest.raises(ffi.Malformed):
            ffi.proof_decode_compressed(enc[:cut])
    with pytest.raises(ffi.Malformed):
        ffi.proof_decode_compressed(enc + b"\0")
    # x = q (with either sign flag)
    for flag in (0, 0x80):
        bad = bytearray(good)
        bad[0:48] = Q.to_bytes(48, "little")
        bad[47] |= flag
        _expect_malformed(bad)
    # an x with no root
    x = _no_root_x()
    with pytest.raises(ValueError):
        ref.g1_deserialize_compressed(x.to_bytes(48, "little"))
    bad = bytearray(good)
    bad[48:96] = x.to_bytes(48, "little")
    _expect_malformed(bad)
    # both flags
    bad = bytearray(good)
    bad[47] |= 0xC0
    _expect_malformed(bad)
    # infinity with x != 0, infinity with the sign bit
    bad = bytearray(good)
    bad[47] = (bad[47] & 0x3F) | 0x40
    _expect_malformed(bad)
    bad = bytearray(good)
    bad[0:48] = bytes(47) + b"\xc0"
    _expect_malformed(bad)
    # a scalar >= r (a.y sits after two compressed points)
    bad = bytearray(good)
    bad[96:128] = R.to_bytes(32, "little")
    _expect_malformed(bad)
    # the canonical infinity record decodes to the uncompressed infinity record
    ok = bytearray(good)
    ok[0:48] = bytes(47) + b"\x40"
    fixed = ffi.proof_decompress(bytes(ok))
    assert fixed[:96] == curve.g1_serialize_unchecked(None)
    assert ffi.proof_compress(fixed) == bytes(ok)


def test_order_three_point_decodes_and_fails_the_subgroup_check():
    """x = 0 without the infinity flag is (0, +-2), a curve point of order 3: decoded, then rejected by
    tp_proof_points_in_subgroup.  The oracle's g1_mul reduces its scalar mod r, so the check is [r - 1]P == -P."""
    two = (0, 2)
    assert curve.g1_is_on_curve(two)
    assert curve.g1_mul(two, R - 1) is None and curve.g1_neg(two) is not None   # [r - 1]P = oo != -P
    assert ref.g1_deserialize_compressed(ref.g1_serialize_compressed(two)) == two
    good = bytearray(ffi.proof_compress(_golden_fixed()))
    for y in (2, Q - 2):
        rec = ref.g1_serialize_compressed((0, y))
        bad = bytearray(good)
        bad[0:48] = rec
        fixed = ffi.proof_decompress(bytes(bad))
        assert curve.g1_deserialize_unchecked(fixed[:96]) == (0, y)
        assert not ffi.proof_points_in_subgroup(fixed)
        assert ffi.proof_compress(fixed) == bytes(bad)


def test_decompressed_proofs_agree_with_the_reference_decoder():
    """every accepted compressed point of a perturbed block is the reference's point, every reference rejection is
    the library's"""
    rnd = random.Random(7)
    good = ffi.proof_compress(_golden_fixed())
    for _ in range(40):
        bad = bytearray(good)
        pos = rnd.randrange(48)
        bad[pos] ^= 1 << rnd.randrange(8)
        try:
            pt = ref.g1_deserialize_compressed(bytes(bad[:48]))
        except ValueError:
            _expect_malformed(bad)
            continue
        fixed = ffi.proof_decompress(bytes(bad))
        assert curve.g1_deserialize_unchecked(fixed[:96]) == pt


def test_compressed_codec_is_canonical_under_random_corruption():
    """Whatever bytes come in, tp_proof_decode_compressed either rejects them or accepts an encoding that re-encodes
    to exactly the same bytes.  A flipped sign bit is the valid encoding of -P and must come back unchanged."""
    rnd = random.Random(2025)
    accepted = rejected = 0
    for name in sorted(PROOFS):
        raw = bytes.fromhex(PROOFS[name]["proof_hex"])
        enc = ffi.proof_encode_compressed(*ffi.proof_decode(raw))
        for _ in range(40):
            bad = bytearray(enc)
            for _ in range(rnd.choice([1, 1, 2, 5])):
                pos = rnd.randrange(len(bad))
                bad[pos] ^= 1 << rnd.randrange(8)
            try:
                fixed, pis = ffi.proof_decode_compressed(bytes(bad))
            except ffi.Malformed:
                rejected += 1
                continue
            accepted += 1
            assert ffi.proof_encode_compressed(fixed, pis) == bytes(bad)
        flipped = bytearray(enc)
        flipped[47] ^= 0x80
        fixed, pis = ffi.proof_decode_compressed(bytes(flipped))
        a = curve.g1_deserialize_unchecked(fixed[:96])
        assert a == curve.g1_neg(curve.g1_deserialize_unchecked(raw[:96]))
        assert ffi.proof_encode_compressed(fixed, pis) == bytes(flipped)
    assert accepted > 0 and rejected > 0


def test_argument_errors():
    fixed = _golden_fixed()
    with pytest.raises(ffi.TyplonkError) as e:
        ffi.proof_encode_compressed(fixed, b"\xff" * 32)          # Montgomery limbs >= r
    assert e.value.code == 1
    assert ffi.proof_encode_compressed(fixed, b"") == ffi.proof_compress(fixed) + bytes(8)
    n = struct.unpack("<Q", ffi.proof_encode_compressed(fixed, b"")[848:856])[0]
    assert n == 0


ARK = os.path.join(GOLD, "arkworks_vectors.json")


@pytest.mark.skipif(not os.path.exists(ARK) or "g1_generator_compressed" not in open(ARK).read(),
                    reason="no arkworks compressed vectors yet: run tools/arkworks_dump/run.sh where cargo exists")
def test_arkworks_compressed_vectors():
    vec = json.load(open(ARK))
    g = curve.G1_GEN
    g17 = curve.g1_mul(g, 17)
    assert ref.g1_serialize_compressed(g).hex() == vec["g1_generator_compressed"]
    assert ref.g1_serialize_compressed(g17).hex() == vec["g1_17_compressed"]
    assert ref.g1_serialize_compressed(curve.g1_neg(g17)).hex() == vec["g1_minus_17_compressed"]
    assert ref.g1_serialize_compressed(None).hex() == vec["g1_zero_compressed"]
    tau = rng.fr_rand_stream(1, 1)[0]
    assert ref.g2_serialize_compressed(curve.G2_GEN).hex() == vec["g2_generator_compressed"]
    assert ref.g2_serialize_compressed(curve.g2_mul(curve.G2_GEN, tau)).hex() == vec["g2_tau_seed_1_compressed"]
    raw = bytes.fromhex(PROOFS["readme_pythagoras_3_4_5"]["proof_hex"])
    assert ffi.proof_encode_compressed(*ffi.proof_decode(raw)).hex() == vec["readme_pythagoras_3_4_5_proof_compressed"]
