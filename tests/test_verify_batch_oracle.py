"""CPU: the folded check of tp_verify_batch (csrc/verify_batch.cu) restated with the oracle -- the random weights
(Blake2b-512 of the tag, n, the circuit's commitments and every proof, then StdRng::from_seed / Fr::rand) and the
scalars of L and R over the batch's base set, checked against the six KZG equations written out with the oracle's
linearisation_commitment.  Honest batches pass, a dishonest proof and a cancelling pair fail."""
import hashlib

import pytest

from oracle.pyoracle import builder as obuilder, curve, kzg as okzg, plonk as oplonk, rng
from oracle.pyoracle.fields import R_MOD as M, fr_inv

TAU = rng.fr_rand_stream(1, 1)[0]
BLINDERS = rng.fr_rand_stream(2, 9)
TAG = b"typlonk-verify-batch-v1"


def circuit_pythagoras(inputs):
    a, b, c = inputs
    a = a.clone() * a
    b = b.clone() * b
    c = c.clone() * c
    d = a + b
    d.assert_eq(c)


def circuit_additive(inputs):
    a, b, c, d, e = inputs
    x = (c + d) + e
    a = a + b
    a.assert_eq(x)


def circuit_mul_chain(inputs):
    x, y = inputs
    for _ in range(13):
        x = x * y.clone()


def circuit_commitments(oc):
    return list(oc.fixed_commitments) + list(oc.copy_constrains.sigma_commitments(oc.srs, oc.domain))


def weights(oc, proofs):
    """rho[k][i], i = 0..5 (a, b, c, z, z-omega, r), from the hash of everything tp_verify_batch receives."""
    h = hashlib.blake2b(digest_size=64)
    h.update(TAG)
    h.update(oc.domain.size.to_bytes(8, "little"))
    for c in circuit_commitments(oc):
        h.update(curve.g1_serialize_unchecked(c))
    for p in proofs:
        h.update(p.to_bytes())   # 1472-byte block | u64 count | canonical public inputs
    r = rng.StdRng(h.digest()[:32])
    return [[rng.fr_rand(r) for _ in range(6)] for _ in proofs]


def parse(p):
    ws = [p.a[1][0], p.b[1][0], p.c[1][0], p.z[0], p.zw[0], p.r[0]]
    ys = [p.a[1][1], p.b[1][1], p.c[1][1], p.z[1], p.zw[1], 0]   # r is opened to the value the verifier requires
    coms = [p.a[0], p.b[0], p.c[0], p.z_commitment]
    return ws, ys, coms


def folded_table(oc, proofs, rhos):
    """L and R as the library assembles them: one MSM each over the shared bases and 13 points per proof."""
    n = oc.domain.size
    omega = oc.domain.element(1)
    q_l, q_r, q_o, q_m, q_c = oc.fixed_commitments
    sigma3 = circuit_commitments(oc)[7]
    shared_pts = [q_l, q_r, q_o, q_m, q_c, sigma3, okzg.identity(oc.srs), curve.G1_GEN]
    shared = [0] * 8
    bases, l_sc, r_sc = [], [], []
    for p, rho in zip(proofs, rhos):
        alpha, beta, gamma, zeta = oplonk._verify_challenges(p)
        assert zeta == p.evaluation_point
        ws, ys, coms = parse(p)
        a, b, c = ys[0], ys[1], ys[2]
        zw = ys[4]
        s1, s2 = oc.copy_constrains.sigma_evals(zeta, oc.domain)[:2]
        zn = pow(zeta, n, M)
        zh = (zn - 1) % M
        l0 = zh * fr_inv(n * (zeta - 1) % M) % M
        l2 = 1
        for k, ev in zip(oc.copy_constrains.cosets, (a, b, c)):
            l2 = l2 * ((ev + beta * k % M * zeta + gamma) % M) % M
        l3 = (a + beta * s1 + gamma) % M * ((b + beta * s2 + gamma) % M) % M
        constant = (alpha * (l3 * (c + gamma) % M * zw % M) + l0 * alpha * alpha) % M   # public inputs are all zero
        x = [zeta, zeta, zeta, zeta, zeta * omega % M, zeta]
        bases += ws + coms + list(p.t)
        l_sc += list(rho) + [0] * 7
        r_sc += [rho[i] * x[i] % M for i in range(6)]
        r_sc += [rho[0], rho[1], rho[2], (rho[3] + rho[4] + rho[5] * (l2 * alpha + l0 * alpha * alpha)) % M]
        r_sc += [-rho[5] * zh % M, -rho[5] * zh * zn % M, -rho[5] * zh * zn * zn % M]
        contrib = [rho[5] * a, rho[5] * b, -rho[5] * c, rho[5] * a * b, rho[5],
                   -rho[5] * l3 * alpha * beta * zw, -rho[5] * constant, -sum(r * y for r, y in zip(rho, ys))]
        shared = [(s + t) % M for s, t in zip(shared, contrib)]
    keep = [i for i, pt in enumerate(shared_pts) if pt is not None] + [8 + i for i, pt in enumerate(bases) if pt is not None]
    allb = shared_pts + bases
    L = curve.g1_msm([allb[i] for i in keep], [([0] * 8 + l_sc)[i] for i in keep])
    R = curve.g1_msm([allb[i] for i in keep], [(shared + r_sc)[i] for i in keep])
    return L, R


def folded_direct(oc, proofs, rhos):
    """The same sums from the six KZG equations e(W, tau) = e(x W + C - y G, 1), C_5 = linearisation_commitment."""
    omega = oc.domain.element(1)
    L = R = None
    for p, rho in zip(proofs, rhos):
        alpha, beta, gamma, zeta = oplonk._verify_challenges(p)
        ws, ys, coms = parse(p)
        r_com = oplonk.linearisation_commitment(oc, ys[:3], p.z_commitment, (ys[3], ys[4]), zeta, p.t, (alpha, beta, gamma), 0)
        cs = coms[:3] + [coms[3], coms[3], r_com]
        x = [zeta] * 4 + [zeta * omega % M, zeta]
        for i in range(6):
            L = curve.g1_add(L, curve.g1_mul(ws[i], rho[i]))
            term = curve.g1_sub(curve.g1_add(curve.g1_mul(ws[i], x[i]), cs[i]), curve.g1_mul(curve.G1_GEN, ys[i]))
            R = curve.g1_add(R, curve.g1_mul(term, rho[i]))
    return L, R


def passes(oc, L, R):
    return curve.pairing_product_is_one([(L, oc.srs.g2s), (curve.g1_neg(R), oc.srs.g2)])


CIRCUITS = {
    "pythagoras": (circuit_pythagoras, 3, lambda k: [3, 4, 5]),
    "additive": (circuit_additive, 5, lambda k: [2 + k, 7, 2, 3 + k, 4]),
    "mul_chain_13": (circuit_mul_chain, 2, lambda k: [3 + k, 5]),
}


@pytest.mark.parametrize("name", sorted(CIRCUITS))
def test_honest_batch_passes_the_folded_check(name):
    run, n_inputs, inputs = CIRCUITS[name]
    oc = obuilder.compile_circuit(run, n_inputs, TAU)
    proofs = [oplonk.prove(oc, inputs(k), [0], rng.fr_rand_stream(100 + k, 9)) for k in range(3)]
    rhos = weights(oc, proofs)
    L, R = folded_table(oc, proofs, rhos)
    assert (L, R) == folded_direct(oc, proofs, rhos)
    assert passes(oc, L, R)


def test_dishonest_proof_fails_the_folded_check():
    oc = obuilder.compile_circuit(circuit_pythagoras, 3, TAU)
    proofs = [oplonk.prove(oc, [3, 4, 5], [0], BLINDERS), oplonk.prove(oc, [3, 4, 6], [0], BLINDERS)]   # builder/test.rs:31-37
    rhos = weights(oc, proofs)
    L, R = folded_table(oc, proofs, rhos)
    assert (L, R) == folded_direct(oc, proofs, rhos)
    assert not passes(oc, L, R)


D = curve.g1_mul(curve.G1_GEN, 0x1234567)


def cancelling_pair(fixed: bytes):
    """Two copies of one proof's 1472-byte block with a's witness W replaced by W + D in one and W - D in the other.
    The witnesses are not in the transcript, so both keep their challenge point; weighted equally the two errors cancel."""
    w = curve.g1_deserialize_unchecked(fixed[96:192])
    plus = fixed[:96] + curve.g1_serialize_unchecked(curve.g1_add(w, D)) + fixed[192:]
    minus = fixed[:96] + curve.g1_serialize_unchecked(curve.g1_sub(w, D)) + fixed[192:]
    return plus, minus


def test_cancelling_pair_fails_with_the_derived_weights():
    oc = obuilder.compile_circuit(circuit_mul_chain, 2, TAU)
    p = oplonk.prove(oc, [3, 5], [0], BLINDERS)
    plus, minus = cancelling_pair(p.to_bytes()[:1472])
    w = p.a[1][0]
    assert curve.g1_deserialize_unchecked(plus[96:192]) == curve.g1_add(w, D)
    pa = oplonk.Proof(**{**p.__dict__, "a": (p.a[0], (curve.g1_add(w, D), p.a[1][1]))})
    pb = oplonk.Proof(**{**p.__dict__, "a": (p.a[0], (curve.g1_sub(w, D), p.a[1][1]))})
    assert pa.to_bytes()[:1472] == plus and pb.to_bytes()[:1472] == minus
    assert not oplonk.verify(oc, pa) and not oplonk.verify(oc, pb)
    ones = [[1] * 6, [1] * 6]
    assert passes(oc, *folded_table(oc, [pa, pb], ones))        # equal weights: the errors cancel
    rhos = weights(oc, [pa, pb])
    L, R = folded_table(oc, [pa, pb], rhos)
    assert (L, R) == folded_direct(oc, [pa, pb], rhos)
    assert not passes(oc, L, R)
