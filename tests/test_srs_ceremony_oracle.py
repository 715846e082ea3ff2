"""SRS ceremony algebra on the host (csrc/srs_ceremony.cu): the randomised check tp_srs_verify runs, restated on the
oracle's curve arithmetic, and the host-only link check tp_srs_update_check on oracle-made points."""
import random

import pytest

import wire_compressed_ref as ref
from oracle.pyoracle import curve, fields, kzg as okzg
from typlonk_b200 import ffi, field as F

Q, R = fields.Q_MOD, fields.R_MOD
TAU = 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF
S = 0x0FEDCBA987654321FEDCBA987654321FEDCBA98765432


def _powers_check(g1, g2, g2s, rho):
    """tp_srs_verify's pairing step: M = sum rho^i g1[i], L = M - rho^(n-1) g1[n-1], D = M - g1[0];
    e(rho L, g2s) e(-D, g2) == 1"""
    n = len(g1)
    m = curve.g1_msm(g1, [pow(rho, i, R) for i in range(n)])
    l = curve.g1_sub(m, curve.g1_mul(g1[n - 1], pow(rho, n - 1, R)))
    d = curve.g1_sub(m, g1[0])
    return curve.pairing_product_is_one([(curve.g1_mul(l, rho), g2s), (curve.g1_neg(d), g2)])


def _srs_check(g1, g2, g2s, rho):
    """the whole verdict for points already known to lie in their groups"""
    return g1[0] == curve.G1_GEN and g2 == curve.G2_GEN and g2s is not None and _powers_check(g1, g2, g2s, rho)


def _g2_abi(pt):
    return F.g2_to_abi(None if pt is None else ((pt[0].a, pt[0].b), (pt[1].a, pt[1].b)))


def _off_subgroup_g1(rnd):
    """a point of y^2 = x^3 + 4 from a random x: almost surely outside G1 ([r - 1]P != -P; g1_mul reduces mod r)"""
    while True:
        x = rnd.randrange(1, Q)
        y = ref._sqrt((x ** 3 + 4) % Q)
        if y is not None and curve.g1_mul((x, y), R - 1) != curve.g1_neg((x, y)):
            return (x, y)


def _off_subgroup_g2(rnd):
    while True:
        x = curve.Fq2(rnd.randrange(Q), rnd.randrange(Q))
        y = ref._fq2_sqrt(x * x * x + curve.B2)
        if y is not None and curve.g2_mul((x, y), R - 1) != curve.g2_neg((x, y)):
            return (x, y)


@pytest.mark.parametrize("n", [8, 13, 16])
def test_powers_check_accepts_powers_and_rejects_each_kind_of_damage(n):
    rnd = random.Random(n)
    srs = okzg.Srs.from_secret(TAU, n - 3)
    g1, g2, g2s = srs.g1, srs.g2, srs.g2s
    assert len(g1) == n
    rho = rnd.randrange(1, R)
    assert _srs_check(g1, g2, g2s, rho)
    i = rnd.randrange(1, n - 1)
    swapped = list(g1)
    swapped[i], swapped[i + 1] = swapped[i + 1], swapped[i]
    assert not _srs_check(swapped, g2, g2s, rho)
    doubled = list(g1)
    doubled[i] = curve.g1_mul(doubled[i], 2)
    assert not _srs_check(doubled, g2, g2s, rho)
    last = list(g1)
    last[n - 1] = curve.g1_add(last[n - 1], curve.G1_GEN)
    assert not _srs_check(last, g2, g2s, rho)
    assert not _srs_check(g1, g2, curve.g2_mul(curve.G2_GEN, TAU + 1), rho)
    # every point times 3: still a chain with ratio tau, which the pairing alone accepts -- P_0 = G is what rejects it
    scaled = [curve.g1_mul(p, 3) for p in g1]
    assert _powers_check(scaled, g2, g2s, rho)
    assert not _srs_check(scaled, g2, g2s, rho)


def test_powers_check_after_contributions():
    """[s^i] [tau^i] G is the SRS of tau s, and the check accepts it"""
    n = 10
    srs = okzg.Srs.from_secret(TAU, n - 3)
    g1 = [curve.g1_mul(p, pow(S, i, R)) for i, p in enumerate(srs.g1)]
    g2s = curve.g2_mul(srs.g2s, S)
    assert g1 == okzg.Srs.from_secret(TAU * S, n - 3).g1
    assert _srs_check(g1, srs.g2, g2s, 987654321)


def _link(prev_tau, s):
    prev = curve.g1_mul(curve.G1_GEN, prev_tau)
    nxt = curve.g1_mul(curve.G1_GEN, prev_tau * s)
    return F.g1_to_abi(prev), F.g1_to_abi(nxt), _g2_abi(curve.g2_mul(curve.G2_GEN, s))


def test_update_check_accepts_the_honest_link():
    assert ffi.srs_update_check(*_link(TAU, S))
    assert ffi.srs_update_check(*_link(1, S))


def test_update_check_rejects_bad_links():
    rnd = random.Random(7)
    prev, nxt, pub = _link(TAU, S)
    assert not ffi.srs_update_check(prev, nxt, _g2_abi(curve.g2_mul(curve.G2_GEN, S + 1)))   # a wrong s
    assert not ffi.srs_update_check(nxt, prev, pub)                                          # the link backwards
    assert not ffi.srs_update_check(prev, nxt, _g2_abi(None))                                # identity pubkey
    assert ffi.srs_update_check(prev, prev, _g2_abi(curve.G2_GEN))       # s = 1: a valid, if useless, link
    inf = F.g1_to_abi(None)
    assert not ffi.srs_update_check(inf, inf, pub)                                           # infinity on both sides
    # G1 points outside the subgroup, on either side
    bad = F.g1_to_abi(_off_subgroup_g1(rnd))
    assert not ffi.srs_update_check(bad, nxt, pub)
    assert not ffi.srs_update_check(prev, bad, pub)
    # off the curve, and a non-canonical coordinate
    x, y = curve.g1_mul(curve.G1_GEN, TAU)
    assert not ffi.srs_update_check(F.g1_to_abi((x, (y + 1) % Q)), nxt, pub)
    noncanon = bytearray(prev)
    noncanon[0:48] = (int.from_bytes(prev[0:48], "little") + Q).to_bytes(48, "little")
    assert not ffi.srs_update_check(bytes(noncanon), nxt, pub)
    # a pubkey on the twist but outside G2
    assert not ffi.srs_update_check(prev, nxt, _g2_abi(_off_subgroup_g2(rnd)))
    with pytest.raises(ffi.TyplonkError) as e:
        ffi.srs_update_check(None, nxt, pub)
    assert e.value.code == 1
