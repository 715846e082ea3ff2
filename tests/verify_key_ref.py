"""Reference restatement of the verification-key wire form (include/typlonk_b200.h, "verification keys"), built from
the oracle alone: sigma_1, sigma_2 from the oracle's permutation (permutation/src/lib.rs:101-194), the commitments
from its KZG over Srs::from_secret(tau).

    "TPVK" | u32 LE version = 1 | u64 LE n | 3 x Fr k | 9 x G1 | G2 g2 | G2 g2s | Vec<Fr> sigma_1 | Vec<Fr> sigma_2

Fr = 32 B LE canonical, G1 = 96 B and G2 = 192 B ark-serialize 0.3 uncompressed, Vec = u64 LE length + items.  The nine
G1 points are q_l q_r q_o q_m q_c, the three sigma commitments and identity = srs[0]."""
from oracle.pyoracle import builder, kzg
from oracle.pyoracle.curve import g1_serialize_unchecked

TAG = b"TPVK"
VERSION = 1
HEAD = 1376
G1_NAMES = ["q_l", "q_r", "q_o", "q_m", "q_c", "sigma_1 commitment", "sigma_2 commitment", "sigma_3 commitment",
            "identity"]


def layout(n: int) -> dict:
    """Byte offset of every field of a key with n rows, and the total size."""
    off = {"tag": 0, "version": 4, "n": 8, "k": 16, "g1": 112, "g2": 976, "g2s": 1168, "sigma_1_len": 1360,
           "sigma_1": 1368}
    off["sigma_2_len"] = off["sigma_1"] + 32 * n
    off["sigma_2"] = off["sigma_2_len"] + 8
    off["size"] = off["sigma_2"] + 32 * n
    assert off["size"] == HEAD + 64 * n
    return off


def fr_bytes(v: int) -> bytes:
    return v.to_bytes(32, "little")


def g2_wire(pt) -> bytes:
    x, y = pt
    return b"".join(v.to_bytes(48, "little") for v in (x.a, x.b, y.a, y.b))


def sigma_coefficients(oc):
    """sigma_1, sigma_2, sigma_3 in coefficient form, padded to n (the oracle strips trailing zeros)."""
    n = oc.domain.size
    return [list(p) + [0] * (n - len(p)) for p in oc.copy_constrains.sigma_polys(oc.domain)]


def vk_bytes_of(oc) -> bytes:
    n = oc.domain.size
    sig = sigma_coefficients(oc)
    points = list(oc.fixed_commitments) + [kzg.commit(oc.srs, s) for s in sig] + [kzg.identity(oc.srs)]
    out = bytearray(TAG + VERSION.to_bytes(4, "little") + n.to_bytes(8, "little"))
    out += b"".join(fr_bytes(k) for k in oc.copy_constrains.cosets)
    out += b"".join(g1_serialize_unchecked(p) for p in points)
    out += g2_wire(oc.srs.g2) + g2_wire(oc.srs.g2s)
    for s in sig[:2]:
        out += n.to_bytes(8, "little") + b"".join(fr_bytes(c) for c in s)
    return bytes(out)


def vk_bytes(run, n_inputs: int, tau: int) -> bytes:
    """The key of `run` compiled under tau, as the library must write it."""
    return vk_bytes_of(builder.compile_circuit(run, n_inputs, tau))
