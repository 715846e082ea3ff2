"""ORACLE (test infrastructure only).

Restatement of proof format v2 (DESIGN.md, "Proof format v2") on the oracle's poly, kzg and curve code:
public gates, the bound transcript, one batched opening at zeta and one at zeta*omega, the 1368-byte key and the
O(l) verifier.  Gates, copy constraints, grand product and quotient are v1's (plonk.py).
"""
import hashlib
from dataclasses import dataclass
from typing import List

from . import kzg, poly
from .builder import GATE_ROWS, BuildVar, CompiledCircuit, ComputeVar, Context
from .curve import (G1_GEN, g1_add, g1_is_on_curve, g1_mul, g1_neg, g1_serialize_unchecked, g1_sub,
                    pairing_product_is_one)
from .fields import R_MOD, fr_inv
from .plonk import linearisation_poly, quotient_polynomial

M = R_MOD
GATE_PUBLIC = "Public"
ROWS = dict(GATE_ROWS, **{GATE_PUBLIC: (1, 0, 0, 0, 0)})
DOMAIN_TAG = b"typlonk-plonk-v2"
VK_TAG = b"TPK2"
VK_BYTES = 1368
PROOF_BYTES = 1056


class ZetaInDomain(ValueError):
    """zeta^n = 1: L_i(zeta) is undefined (the prover gives up, the verifier rejects)."""


# ---- circuit ---------------------------------------------------------------------------------------------------------

def trace_public(run, n_inputs: int, n_public: int):
    """The tracer with public gates: rows 0..l-1 hold input i at cell (0, i), selectors q_l = 1; later uses of x_i get
    copy constraints through the existing rule for already-placed operands."""
    assert 0 <= n_public <= n_inputs
    ctx = Context()
    inputs = [BuildVar.input(ctx) for _ in range(n_inputs)]
    for i in range(n_public):
        j = ctx.add_gate(GATE_PUBLIC)
        ctx.add_var(inputs[i].id, (0, j))
    run(inputs)
    gates, permutation = ctx.finish()
    return gates, permutation.build(len(gates))


@dataclass
class CircuitV2:
    oc: CompiledCircuit
    n_public: int


def compile_circuit(run, n_inputs: int, n_public: int, tau: int) -> CircuitV2:
    """builder.compile_circuit with the public gates in front."""
    from .poly import Domain, interpolate
    gates, perm = trace_public(run, n_inputs, n_public)
    domain = Domain(len(gates))
    srs = kzg.Srs.from_secret(tau, domain.size)
    cols = [[ROWS[g][k] for g in gates] for k in range(5)]
    selectors = [interpolate(c, domain) for c in cols]
    commitments = [kzg.commit(srs, p) for p in selectors]
    oc = CompiledCircuit(run, n_inputs, selectors, commitments, perm.compile(), srs, domain, len(gates), gates)
    return CircuitV2(oc, n_public)


def witness_columns(circuit: CircuitV2, inputs, blinders):
    """witness_columns with a = x_i, b = c = 0 in the public rows."""
    oc = circuit.oc
    rows = oc.rows
    advice = [[], [], []]
    for i in range(circuit.n_public):
        for col, v in zip(advice, (inputs[i] % M, 0, 0)):
            col.append(v)
    oc.run([ComputeVar(v, advice) for v in inputs])
    out = []
    for k, col in enumerate(advice):
        col = col[: rows - 3] + [0] * max(0, rows - 3 - len(col))
        out.append(col + [b % M for b in blinders[3 * k: 3 * k + 3]])
    return out


# ---- key -------------------------------------------------------------------------------------------------------------

def g2_wire(pt) -> bytes:
    x, y = pt
    return b"".join(v.to_bytes(48, "little") for v in (x.a, x.b, y.a, y.b))


def sigma_commitments(oc):
    return [kzg.commit(oc.srs, p) for p in oc.copy_constrains.sigma_polys(oc.domain)]


def vk_bytes(circuit: CircuitV2) -> bytes:
    """"TPK2" | u32 1 | u64 n | u64 l | 3 Fr k | 9 G1 (q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 srs[0]) | G2 g2 |
    G2 g2s."""
    oc = circuit.oc
    n = oc.domain.size
    points = list(oc.fixed_commitments) + sigma_commitments(oc) + [kzg.identity(oc.srs)]
    out = VK_TAG + (1).to_bytes(4, "little") + n.to_bytes(8, "little") + circuit.n_public.to_bytes(8, "little")
    out += b"".join(k.to_bytes(32, "little") for k in oc.copy_constrains.cosets)
    out += b"".join(g1_serialize_unchecked(p) for p in points)
    out += g2_wire(oc.srs.g2) + g2_wire(oc.srs.g2s)
    assert len(out) == VK_BYTES
    return out


# ---- transcript ------------------------------------------------------------------------------------------------------

def _h(data: bytes) -> bytes:
    return hashlib.blake2b(data, digest_size=64).digest()


class Transcript:
    def __init__(self, vk: bytes, public_values):
        self.s = _h(DOMAIN_TAG + _h(vk) + len(public_values).to_bytes(8, "little") +
                    b"".join((v % M).to_bytes(32, "little") for v in public_values))

    def absorb(self, label: bytes, points=(), scalars=()):
        data = b"".join(g1_serialize_unchecked(p) for p in points) + b"".join(s.to_bytes(32, "little") for s in scalars)
        self.s = _h(self.s + label + data)

    def squeeze(self, i: int) -> int:
        return int.from_bytes(_h(self.s + b"challenge" + bytes([i])), "little") % M


# ---- proof -----------------------------------------------------------------------------------------------------------

@dataclass
class ProofV2:
    points: List  # [a] [b] [c] [z] [t0] [t1] [t2] [W_zeta] [W_zeta_omega]
    evals: List[int]  # a b c sigma_1 sigma_2 z(zeta omega)
    public_values: List[int]

    def block(self) -> bytes:
        return (b"".join(g1_serialize_unchecked(p) for p in self.points) +
                b"".join(v.to_bytes(32, "little") for v in self.evals))

    def to_bytes(self) -> bytes:
        return (self.block() + len(self.public_values).to_bytes(8, "little") +
                b"".join(v.to_bytes(32, "little") for v in self.public_values))


def pi_column(public_values, n):
    return [(-v) % M for v in public_values] + [0] * (n - len(public_values))


def prove(circuit: CircuitV2, inputs, blinders) -> ProofV2:
    oc = circuit.oc
    cols = witness_columns(circuit, inputs, blinders)
    return prove_columns(circuit, cols)


def prove_columns(circuit: CircuitV2, cols, vk=None) -> ProofV2:
    oc = circuit.oc
    domain, srs = oc.domain, oc.srs
    n = domain.size
    w = domain.element(1)
    publics = cols[0][: circuit.n_public]
    tr = Transcript(vk or vk_bytes(circuit), publics)
    pi_poly = poly.interpolate(pi_column(publics, n), domain)
    advice = [poly.interpolate(c, domain) for c in cols]
    coms = [kzg.commit(srs, p) for p in advice]
    tr.absorb(b"abc", coms)
    beta, gamma = tr.squeeze(0), tr.squeeze(1)
    evals = oc.copy_constrains.prove([domain.fft(p) for p in advice], beta, gamma)
    evals.pop()
    acc_shifted = poly.interpolate(evals[1:] + evals[:1], domain)
    acc = poly.interpolate(evals, domain)
    zc = kzg.commit(srs, acc)
    tr.absorb(b"z", [zc])
    alpha = tr.squeeze(0)
    t = quotient_polynomial(oc, advice, (acc, acc_shifted), (alpha, beta, gamma), pi_poly, False)
    tc = [kzg.commit(srs, s) for s in t]
    tr.absorb(b"t", tc)
    zeta = tr.squeeze(0)
    if pow(zeta, n, M) == 1:
        raise ZetaInDomain()
    sig = oc.copy_constrains.sigma_polys(domain)
    opened = advice + sig[:2]
    ys = [poly.evaluate(p, zeta) for p in opened]
    zw = poly.evaluate(acc, zeta * w % M)
    tr.absorb(b"evals", scalars=ys + [zw])
    v = tr.squeeze(0)
    r = linearisation_poly(oc, ys[:3], (poly.evaluate(acc, zeta), zw), acc, (alpha, beta, gamma), zeta, t,
                           poly.evaluate(pi_poly, zeta))
    big = poly.strip(r)
    vj = 1
    for p, y in zip(opened, ys):
        vj = vj * v % M
        big = poly.add(big, poly.scale(poly.sub(p, [y]), vj))
    w_zeta = kzg.open_at(srs, poly.strip(big), zeta)[0]
    w_zw = kzg.open_at(srs, acc, zeta * w % M)[0]
    return ProofV2(coms + [zc] + tc + [w_zeta, w_zw], ys + [zw], [x % M for x in publics])


# ---- verifier --------------------------------------------------------------------------------------------------------

def _lagrange_at(n, omega, zeta, count):
    """L_i(zeta) = omega^i (zeta^n - 1) / (n (zeta - omega^i)), i < count, with one inversion."""
    zh = (pow(zeta, n, M) - 1) % M
    dens, wi = [], 1
    for _ in range(count):
        dens.append(n * (zeta - wi) % M)
        wi = wi * omega % M
    prod, acc = 1, []
    for d in dens:
        acc.append(prod)
        prod = prod * d % M
    inv = fr_inv(prod)
    out = [0] * count
    for i in range(count - 1, -1, -1):
        out[i] = inv * acc[i] % M
        inv = inv * dens[i] % M
    wi, res = 1, []
    for i in range(count):
        res.append(wi * zh % M * out[i] % M)
        wi = wi * omega % M
    return res


def parse_vk(vk: bytes):
    from .curve import g1_deserialize_unchecked
    n = int.from_bytes(vk[8:16], "little")
    ell = int.from_bytes(vk[16:24], "little")
    ks = [int.from_bytes(vk[24 + 32 * i: 56 + 32 * i], "little") for i in range(3)]
    pts = [g1_deserialize_unchecked(vk[120 + 96 * i: 216 + 96 * i]) for i in range(9)]
    return n, ell, ks, pts


def verify(vk: bytes, srs: kzg.Srs, proof: ProofV2, public_values, use_trapdoor=False) -> bool:
    """O(l) verifier.  The key is the wire bytes; srs supplies g2, g2s (and the secret for the trapdoor variant)."""
    n, ell, ks, pts = parse_vk(vk)
    ql, qr, qo, qm, qc, s1, s2, s3, g = pts
    if len(public_values) != ell or len(proof.public_values) != ell:
        return False
    if any(v >= M for v in public_values) or list(public_values) != list(proof.public_values):
        return False
    if len(proof.points) != 9 or len(proof.evals) != 6 or any(not (0 <= e < M) for e in proof.evals):
        return False
    if any(p is not None and not g1_is_on_curve(p) for p in proof.points):
        return False
    ca, cb, cc, cz, t0, t1, t2, wz, wzw = proof.points
    a, b, c, sb1, sb2, zw = proof.evals
    tr = Transcript(vk, public_values)
    tr.absorb(b"abc", [ca, cb, cc])
    beta, gamma = tr.squeeze(0), tr.squeeze(1)
    tr.absorb(b"z", [cz])
    alpha = tr.squeeze(0)
    tr.absorb(b"t", [t0, t1, t2])
    zeta = tr.squeeze(0)
    if pow(zeta, n, M) == 1:
        return False
    tr.absorb(b"evals", scalars=proof.evals)
    v = tr.squeeze(0)
    tr.absorb(b"w", [wz, wzw])
    u = tr.squeeze(0)
    from .fields import root_of_unity
    omega = root_of_unity(n)
    lag = _lagrange_at(n, omega, zeta, max(ell, 1))
    pi_bar = sum((-x) * l for x, l in zip(public_values, lag)) % M
    zn = pow(zeta, n, M)
    zh = (zn - 1) % M
    l0 = _lagrange_at(n, omega, zeta, 1)[0]
    l2 = 1
    for k, ev in zip(ks, (a, b, c)):
        l2 = l2 * ((ev + k * beta % M * zeta + gamma) % M) % M
    perm_ab = (a + beta * sb1 + gamma) % M * ((b + beta * sb2 + gamma) % M) % M
    ab_zw = alpha * perm_ab % M * zw % M
    const = (pi_bar - ab_zw * (gamma + c) - alpha * alpha % M * l0) % M
    terms = [(ql, a), (qr, b), (qo, (-c) % M), (qm, a * b % M), (qc, 1),
             (cz, (alpha * l2 + alpha * alpha % M * l0) % M), (s3, (-ab_zw * beta) % M),
             (t0, (-zh) % M), (t1, (-zh * zn) % M), (t2, (-zh * zn % M * zn) % M), (g, const)]
    vs = [pow(v, j, M) for j in range(1, 6)]
    terms += list(zip((ca, cb, cc, s1, s2), vs))
    e_scalar = sum(vj * y for vj, y in zip(vs, (a, b, c, sb1, sb2))) % M
    zeta_w = zeta * omega % M
    # F - E + u([z] - zw G) + zeta W_zeta + u zeta omega W_zeta_omega
    rhs = None
    for p, s in terms + [(g, (-e_scalar) % M), (cz, u), (g, (-u * zw) % M), (wz, zeta), (wzw, u * zeta_w % M)]:
        rhs = g1_add(rhs, g1_mul(p, s))
    lhs = g1_add(wz, g1_mul(wzw, u))
    if use_trapdoor:
        assert srs.secret is not None
        return g1_mul(lhs, srs.secret) == rhs
    return pairing_product_is_one([(lhs, srs.g2s), (g1_neg(rhs), srs.g2)])
