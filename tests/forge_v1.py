"""The forgery that proof format v1 admits (DESIGN.md, "Proof format v2"), built on the oracle: v1 draws zeta from
[a] [b] [c] [z] alone and never hashes [t0] [t1] [t2], so a prover who knows zeta can take t as the constant
Lin(zeta) / Z_H(zeta), which makes r(zeta) = 0 for any witness.  The same construction against v2 has to guess zeta
before committing to t, and the verifier's zeta, drawn after [t], differs."""
from oracle.pyoracle import builder as ob, kzg, plonk_v2 as ov2, poly
from oracle.pyoracle.plonk import M, Proof, generate_challenges, linearisation_poly, transcript

FALSE_INPUTS = [3, 4, 6]   # 3^2 + 4^2 != 6^2


def _forged_t(oc, advice, acc, challenges, zeta, public_eval):
    aev = [poly.evaluate(p, zeta) for p in advice]
    zw = poly.evaluate(acc, zeta * oc.domain.element(1) % M)
    lin0 = linearisation_poly(oc, aev, (poly.evaluate(acc, zeta), zw), acc, challenges, zeta, [[], [], []], public_eval)
    zh = oc.domain.evaluate_vanishing_polynomial(zeta)
    return [[poly.evaluate(lin0, zeta) * pow(zh, M - 2, M) % M], [], []]


def forged_v1_proof(tau, blinders):
    """(compiled circuit, v1 Proof of the false statement 3^2 + 4^2 = 6^2 for the README circuit)."""
    oc = ob.compile_circuit(ob.circuit_pythagoras, 3, tau)
    dom, srs = oc.domain, oc.srs
    cols = ob.witness_columns(oc.run, FALSE_INPUTS, oc.rows, blinders)
    adv = [poly.interpolate(c, dom) for c in cols]
    coms = [kzg.commit(srs, p) for p in adv]
    beta, gamma = generate_challenges(transcript(coms), 2)
    ev = oc.copy_constrains.prove([dom.fft(p) for p in adv], beta, gamma)
    ev.pop()
    acc = poly.interpolate(ev, dom)
    zc = kzg.commit(srs, acc)
    alpha, zeta = generate_challenges(transcript(coms + [zc]), 2)
    t = _forged_t(oc, adv, acc, (alpha, beta, gamma), zeta, 0)
    lin = linearisation_poly(oc, [poly.evaluate(p, zeta) for p in adv],
                             (poly.evaluate(acc, zeta), poly.evaluate(acc, zeta * dom.element(1) % M)), acc,
                             (alpha, beta, gamma), zeta, t, 0)
    ops = [kzg.open_at(srs, p, zeta) for p in adv]
    pf = Proof(a=(coms[0], ops[0]), b=(coms[1], ops[1]), c=(coms[2], ops[2]), z_commitment=zc,
               z=kzg.open_at(srs, acc, zeta), zw=kzg.open_at(srs, acc, zeta * dom.element(1) % M),
               evaluation_point=zeta, t=[kzg.commit(srs, s) for s in t], r=kzg.open_at(srs, poly.strip(lin), zeta),
               public_inputs=[0] * oc.rows)
    return oc, pf


def forged_v2_attempt(tau, blinders, n_public=0):
    """The same construction against v2: zeta is guessed from the transcript before [t] (as if t were 0), t is made
    constant for that guess, and the openings are made at the guess.  Returns (circuit, key bytes, proof)."""
    circuit = ov2.compile_circuit(ob.circuit_pythagoras, 3, n_public, tau)
    oc = circuit.oc
    dom, srs = oc.domain, oc.srs
    n = dom.size
    cols = ov2.witness_columns(circuit, FALSE_INPUTS, blinders)
    publics = cols[0][:n_public]
    vk = ov2.vk_bytes(circuit)
    tr = ov2.Transcript(vk, publics)
    pi_poly = poly.interpolate(ov2.pi_column(publics, n), dom)
    adv = [poly.interpolate(c, dom) for c in cols]
    coms = [kzg.commit(srs, p) for p in adv]
    tr.absorb(b"abc", coms)
    beta, gamma = tr.squeeze(0), tr.squeeze(1)
    ev = oc.copy_constrains.prove([dom.fft(p) for p in adv], beta, gamma)
    ev.pop()
    acc = poly.interpolate(ev, dom)
    zc = kzg.commit(srs, acc)
    tr.absorb(b"z", [zc])
    alpha = tr.squeeze(0)
    guess = ov2.Transcript.__new__(ov2.Transcript)
    guess.s = tr.s
    guess.absorb(b"t", [None, None, None])
    zeta = guess.squeeze(0)
    t = _forged_t(oc, adv, acc, (alpha, beta, gamma), zeta, poly.evaluate(pi_poly, zeta))
    tc = [kzg.commit(srs, s) for s in t]
    sig = oc.copy_constrains.sigma_polys(dom)
    opened = adv + sig[:2]
    ys = [poly.evaluate(p, zeta) for p in opened]
    zw = poly.evaluate(acc, zeta * dom.element(1) % M)
    tr.absorb(b"t", tc)
    tr.absorb(b"evals", scalars=ys + [zw])
    v = tr.squeeze(0)
    r = linearisation_poly(oc, ys[:3], (poly.evaluate(acc, zeta), zw), acc, (alpha, beta, gamma), zeta, t,
                           poly.evaluate(pi_poly, zeta))
    big, vj = poly.strip(r), 1
    for p, y in zip(opened, ys):
        vj = vj * v % M
        big = poly.add(big, poly.scale(poly.sub(p, [y]), vj))
    proof = ov2.ProofV2(coms + [zc] + tc + [kzg.open_at(srs, poly.strip(big), zeta)[0],
                                            kzg.open_at(srs, acc, zeta * dom.element(1) % M)[0]],
                        ys + [zw], publics)
    return circuit, vk, proof
