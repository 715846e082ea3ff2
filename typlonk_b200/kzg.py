"""Host-side mirror of the reference's `kzg` crate API (kzg/src/srs.rs, kzg/src/lib.rs:33-86)
over the CUDA library: same names, argument meaning and error behaviour, so the parity tests
read like the reference's own tests.  Scalars/points at this level are canonical Python ints /
affine (x, y) tuples (None = infinity)."""
import secrets

from . import field as F
from . import ffi
from .ffi import Context, TyplonkError  # noqa: F401


class Srs:
    """kzg/src/srs.rs:8-52.  The G1 powers live on the device."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.handle = handle

    @classmethod
    def from_secret(cls, ctx: Context, s: int, gates: int) -> "Srs":
        """Srs::from_secret (srs.rs:30-34): gates + 3 powers, generated on the GPU."""
        return cls(ctx, ctx.srs_from_secret(F.fr_to_bytes(s), gates))

    @classmethod
    def from_points(cls, ctx: Context, points) -> "Srs":
        return cls(ctx, ctx.srs_upload(b"".join(F.g1_to_packed(p) for p in points)))

    def to_bytes(self, compressed=False) -> bytes:
        """Vec<G1> | G2 | tau G2 in ark-serialize 0.3 uncompressed encoding (tp_srs_serialize; SURVEY.md 8 f4), or
        with compressed points (tp_srs_serialize_compressed: 48 B per G1 point, 96 B per G2 point)."""
        return bytes(self.handle.serialize_compressed() if compressed else self.handle.serialize())

    @classmethod
    def from_bytes(cls, ctx: Context, raw, check=2, compressed=False) -> "Srs":
        """tp_srs_deserialize / tp_srs_deserialize_compressed: validated on the device (check = 2: on the curve and in
        the prime-order subgroup; compressed points are decompressed there too)."""
        if compressed:
            return cls(ctx, ctx.srs_deserialize_compressed(raw, check))
        return cls(ctx, ctx.srs_deserialize(raw, check))

    def contribute(self, s=None):
        """One powers-of-tau contribution (tp_srs_contribute) -> (new Srs, pubkey [s]G2 in the g2_ref() shape).  With
        s = None the secret is drawn from the operating system's CSPRNG and never returned.  This Srs is unchanged."""
        if s is None:
            s = secrets.randbelow(F.R_MOD - 1) + 1
        handle, pub = self.ctx.srs_contribute(self.handle, F.fr_to_bytes(s))
        return Srs(self.ctx, handle), F.g2_from_abi(pub)

    def verify(self) -> bool:
        """tp_srs_verify: g1[i] = [t^i]G for the t with g2s = [t]G2, g2 = the G2 generator, every point in its group."""
        return self.ctx.srs_verify(self.handle)

    def verify_update(self, prev: "Srs", pubkey) -> bool:
        """tp_srs_update_check on g1[1] of `prev` and of this SRS: was this SRS made from `prev` by the contribution
        whose pubkey ([s]G2, g2_ref() shape) is given?"""
        def tau_g1(srs):
            return F.g1_to_abi(F.g1_from_packed(srs.handle.download(1, 1)))
        return ffi.srs_update_check(tau_g1(prev), tau_g1(self), F.g2_to_abi(pubkey))

    def g1_ref(self, offset=0, count=None):
        raw = self.handle.download(offset, count)
        return [F.g1_from_packed(raw[i:i + 96]) for i in range(0, len(raw), 96)]

    def g2_ref(self):
        """srs.rs:46-48, as ((x0, x1), (y0, y1)) canonical ints."""
        return F.g2_from_abi(self.handle.g2()[0])

    def g2s_ref(self):
        """srs.rs:49-51."""
        return F.g2_from_abi(self.handle.g2()[1])

    def __len__(self):
        return len(self.handle)


class KzgScheme:
    """kzg/src/lib.rs:33-86."""

    def __init__(self, srs: Srs):
        self.srs = srs
        self.ctx = srs.ctx

    def commit(self, polynomial):
        """KzgScheme::commit (lib.rs:37-54); polynomial = coefficient list (trailing zeros
        stripped like DensePolynomial).  Raises where the reference's assert fires."""
        coeffs = _strip(polynomial)
        out = self.ctx.commit(self.srs.handle, F.fr_vec_to_bytes(coeffs))
        return F.g1_from_abi(out)

    def open(self, polynomial, z: int):
        """KzgScheme::open (lib.rs:55-64) -> (witness point, evaluation)."""
        coeffs = _strip(polynomial)
        w, y = self.ctx.open(self.srs.handle, F.fr_vec_to_bytes(coeffs), F.fr_to_bytes(z))
        return F.g1_from_abi(w), F.fr_from_bytes(y)

    def verify(self, commitment, opening, z: int) -> bool:
        """KzgScheme::verify (lib.rs:66-81): opening = (witness point, evaluation).  The pairing is O(1) host work
        inside the library (csrc/pairing.h)."""
        w, y = opening
        g2, g2s = self.srs.handle.g2()
        return ffi.kzg_verify(g2, g2s, F.g1_to_abi(commitment), F.g1_to_abi(w), F.fr_to_bytes(y), F.fr_to_bytes(z))

    def identity(self):
        return self.commit([1])


def _strip(p):
    p = [x % F.R_MOD for x in p]
    while p and p[-1] == 0:
        p.pop()
    return p
