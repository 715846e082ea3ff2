"""Reference codec for the compressed wire encodings (ark-serialize 0.3 `serialize` of ark-ec 0.3 short-Weierstrass
points), written directly from the encoding's rules on Python integers, independently of csrc/wire.cu:

- G1, 48 B: canonical x, little-endian; bit 7 of byte 47 set iff y > -y (canonical integers), bit 6 = infinity
  (x = 0, bit 7 clear); both bits set is invalid.  Decoding: x < q, y = (x^3 + 4)^((q+1)/4), y^2 must equal x^3 + 4.
- G2, 96 B: x.c0 | x.c1, the flags in the last byte of x.c1; Fq2's order compares c1 first, then c0.  The square
  root here uses the norm method (a different algorithm from the library's), checked by squaring.

Points are the oracle's: (x, y) canonical integers for G1, (Fq2, Fq2) for G2, None = infinity."""
from oracle.pyoracle.curve import B2, Fq2
from oracle.pyoracle.fields import Q_MOD

Q = Q_MOD
INF, POS = 0x40, 0x80


def _is_positive(y: int) -> bool:
    return y > (-y) % Q


def _fq2_is_positive(y: Fq2) -> bool:
    if y.b != (-y.b) % Q:
        return _is_positive(y.b)
    return _is_positive(y.a)


def _sqrt(a: int):
    y = pow(a, (Q + 1) // 4, Q)
    return y if y * y % Q == a % Q else None


def _fq2_sqrt(a: Fq2):
    """sqrt(a0 + a1 u), u^2 = -1: x0^2 - x1^2 = a0, 2 x0 x1 = a1 with x0^2 = (a0 +- |a|) / 2, |a| = sqrt(a0^2 + a1^2)"""
    if a.b == 0:
        r = _sqrt(a.a)
        if r is not None:
            return Fq2(r, 0)
        r = _sqrt(-a.a % Q)
        return Fq2(0, r) if r is not None else None
    n = _sqrt((a.a * a.a + a.b * a.b) % Q)
    if n is None:
        return None
    inv2 = pow(2, -1, Q)
    for d in ((a.a + n) * inv2 % Q, (a.a - n) * inv2 % Q):
        x0 = _sqrt(d)
        if x0 is not None and x0 != 0:
            x = Fq2(x0, a.b * pow(2 * x0, -1, Q))
            if x * x == a:
                return x
    return None


def g1_serialize_compressed(pt) -> bytes:
    if pt is None:
        out = bytearray(48)
        out[47] = INF
        return bytes(out)
    out = bytearray(pt[0].to_bytes(48, "little"))
    if _is_positive(pt[1]):
        out[47] |= POS
    return bytes(out)


def g1_deserialize_compressed(b: bytes):
    """-> point (None = infinity); ValueError for a record that no point encodes to."""
    if len(b) != 48:
        raise ValueError("length")
    flags = b[47] & 0xC0
    x = int.from_bytes(b[:47] + bytes([b[47] & 0x3F]), "little")
    if flags == INF | POS or x >= Q:
        raise ValueError("flags or x >= q")
    if flags & INF:
        if x:
            raise ValueError("infinity with x != 0")
        return None
    y = _sqrt((x ** 3 + 4) % Q)
    if y is None:
        raise ValueError("no root")
    if _is_positive(y) != bool(flags & POS):
        y = (-y) % Q
    return (x, y)


def g2_serialize_compressed(pt) -> bytes:
    if pt is None:
        out = bytearray(96)
        out[95] = INF
        return bytes(out)
    x, y = pt
    out = bytearray(x.a.to_bytes(48, "little") + x.b.to_bytes(48, "little"))
    if _fq2_is_positive(y):
        out[95] |= POS
    return bytes(out)


def g2_deserialize_compressed(b: bytes):
    if len(b) != 96:
        raise ValueError("length")
    flags = b[95] & 0xC0
    x0 = int.from_bytes(b[:48], "little")
    x1 = int.from_bytes(b[48:95] + bytes([b[95] & 0x3F]), "little")
    if flags == INF | POS or x0 >= Q or x1 >= Q:
        raise ValueError("flags or coordinate >= q")
    if flags & INF:
        if x0 or x1:
            raise ValueError("infinity with x != 0")
        return None
    x = Fq2(x0, x1)
    y = _fq2_sqrt(x * x * x + B2)
    if y is None:
        raise ValueError("no root")
    if _fq2_is_positive(y) != bool(flags & POS):
        y = -y
    return (x, y)


PROOF_LAYOUT = "GGF" "GGF" "GGF" "GGF" "GF" "F" "GGG" "GF"


def proof_block_compress(fixed: bytes) -> bytes:
    """1472-byte uncompressed block (oracle-encoded points) -> 848-byte compressed block."""
    from oracle.pyoracle import curve
    out, p = b"", 0
    for k in PROOF_LAYOUT:
        if k == "G":
            out += g1_serialize_compressed(curve.g1_deserialize_unchecked(fixed[p:p + 96]))
            p += 96
        else:
            out += fixed[p:p + 32]
            p += 32
    return out
