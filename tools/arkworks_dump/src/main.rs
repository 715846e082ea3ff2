//! Writes arkworks-generated known answers for everything the oracle restates from memory (SURVEY.md App. A.4 - A.6):
//! `serialize_unchecked` of G1 points, `StdRng::seed_from_u64`, `Fr::rand`, the challenge chain of
//! plonk/src/proof/challenges.rs, domain elements, whole proofs of the reference's own circuits under the fixed
//! randomness run.sh patches in, and the compressed encoding (`serialize`) of G1 / G2 points and of one proof.  Output: one JSON object (hex strings are little-endian bytes as arkworks writes them).
use ark_bls12_381::{Fr, G1Affine, G2Affine};
use ark_ec::AffineCurve;
use ark_ff::{BigInteger, FftField, PrimeField, UniformRand, Zero};
use ark_poly::{EvaluationDomain, GeneralEvaluationDomain};
use ark_serialize::CanonicalSerialize;
use blake2::{Blake2b, Digest};
use plonk::description::{CircuitDescription, Var};
use rand::{rngs::StdRng, RngCore, SeedableRng};
use std::fmt::Write as _;

fn hex(b: &[u8]) -> String {
    let mut s = String::new();
    for x in b {
        write!(s, "{:02x}", x).unwrap();
    }
    s
}
fn fr_canonical(x: &Fr) -> String {
    hex(&x.into_repr().to_bytes_le())
}
fn fr_montgomery(x: &Fr) -> String {
    // the in-memory limbs (ark_ff::Fp256 .0), what crosses the C ABI
    let mut out = vec![];
    for l in (x.0).0.iter() {
        out.extend_from_slice(&l.to_le_bytes());
    }
    hex(&out)
}
fn g1_unchecked(p: &G1Affine) -> String {
    let mut v = vec![];
    p.serialize_unchecked(&mut v).unwrap();
    hex(&v)
}
fn g1_compressed(p: &G1Affine) -> String {
    let mut v = vec![];
    p.serialize(&mut v).unwrap();
    hex(&v)
}
fn g2_compressed(p: &G2Affine) -> String {
    let mut v = vec![];
    p.serialize(&mut v).unwrap();
    hex(&v)
}

struct Pythagoras;
impl CircuitDescription<3> for Pythagoras {
    fn run<V: Var>(inputs: [V; 3]) {
        let [a, b, c] = inputs;
        let a = a.clone() * a;
        let b = b.clone() * b;
        let c = c.clone() * c;
        let d = a + b;
        d.assert_eq(&c);
    }
}
struct MulChain13;
impl CircuitDescription<2> for MulChain13 {
    fn run<V: Var>(inputs: [V; 2]) {
        let [mut x, y] = inputs;
        for _ in 0..13 {
            x = x * y.clone();
        }
    }
}

fn main() {
    let out_path = std::env::args().nth(1).expect("output path");
    let mut j = String::from("{\n");
    let g = G1Affine::prime_subgroup_generator();
    let g17: G1Affine = g.mul(Fr::from(17u64)).into();
    writeln!(j, "  \"g1_generator_unchecked\": \"{}\",", g1_unchecked(&g)).unwrap();
    writeln!(j, "  \"g1_17_unchecked\": \"{}\",", g1_unchecked(&g17)).unwrap();
    writeln!(j, "  \"g1_zero_unchecked\": \"{}\",", g1_unchecked(&G1Affine::zero())).unwrap();
    // compressed (`serialize`): x with the PositiveY / infinity flags in the top bits of the last byte
    writeln!(j, "  \"g1_generator_compressed\": \"{}\",", g1_compressed(&g)).unwrap();
    writeln!(j, "  \"g1_17_compressed\": \"{}\",", g1_compressed(&g17)).unwrap();
    writeln!(j, "  \"g1_minus_17_compressed\": \"{}\",", g1_compressed(&-g17)).unwrap();
    writeln!(j, "  \"g1_zero_compressed\": \"{}\",", g1_compressed(&G1Affine::zero())).unwrap();
    {
        let h = G2Affine::prime_subgroup_generator();
        let tau = Fr::rand(&mut StdRng::seed_from_u64(1));
        let htau: G2Affine = h.mul(tau).into();
        writeln!(j, "  \"g2_generator_compressed\": \"{}\",", g2_compressed(&h)).unwrap();
        writeln!(j, "  \"g2_tau_seed_1_compressed\": \"{}\",", g2_compressed(&htau)).unwrap();
    }
    // StdRng::seed_from_u64(k): first four u64 draws
    for k in [0u64, 1, 2, 13037422643194131432] {
        let mut rng = StdRng::seed_from_u64(k);
        let v: Vec<String> = (0..4).map(|_| rng.next_u64().to_string()).collect();
        writeln!(j, "  \"stdrng_seed_from_u64_{}\": [{}],", k, v.join(", ")).unwrap();
    }
    // Fr::rand: first nine draws of seeds 1 and 2 (tau and the blinders of every test in the repository)
    for k in [1u64, 2, 3, 4] {
        let mut rng = StdRng::seed_from_u64(k);
        let v: Vec<String> = (0..9).map(|_| format!("\"{}\"", fr_montgomery(&Fr::rand(&mut rng)))).collect();
        writeln!(j, "  \"fr_rand_montgomery_seed_{}\": [{}],", k, v.join(", ")).unwrap();
        let mut rng = StdRng::seed_from_u64(k);
        let v: Vec<String> = (0..9).map(|_| format!("\"{}\"", fr_canonical(&Fr::rand(&mut rng)))).collect();
        writeln!(j, "  \"fr_rand_canonical_seed_{}\": [{}],", k, v.join(", ")).unwrap();
    }
    // the challenge chain of challenges.rs:17-45 over the transcript [17 G] x 3
    {
        let mut data = vec![];
        for _ in 0..3 {
            g17.serialize_unchecked(&mut data).unwrap();
        }
        let hash = Blake2b::digest(&data);
        let mut seed = [0u8; 8];
        seed.copy_from_slice(&hash[0..8]);
        let seed = u64::from_le_bytes(seed);
        let mut rng = StdRng::seed_from_u64(seed);
        let c: Vec<String> = (0..2).map(|_| format!("\"{}\"", fr_montgomery(&Fr::rand(&mut rng)))).collect();
        writeln!(j, "  \"challenge_chain_17G_x3\": {{\"seed\": {}, \"challenges_montgomery\": [{}]}},", seed, c.join(", ")).unwrap();
    }
    // domain: omega_8, the 2^32-th root of unity
    {
        let d = <GeneralEvaluationDomain<Fr>>::new(8).unwrap();
        writeln!(j, "  \"omega_8_canonical\": \"{}\",", fr_canonical(&d.element(1))).unwrap();
        writeln!(j, "  \"two_adic_root_canonical\": \"{}\",", fr_canonical(&Fr::two_adic_root_of_unity())).unwrap();
    }
    // whole proofs of the reference under tau = seed 1, blinders = seed 2 (run.sh), field by field in the order of
    // plonk/src/proof.rs:85-95 -- the repository's canonical proof bytes are exactly this concatenation
    // (SURVEY.md App. A.6): a.com a.W a.y | b | c | z.com z.W z.y zw.W zw.y | point | t0 t1 t2 | r.W r.y
    let circuit = Pythagoras::build();
    let proof = circuit.prove([3, 4, 5], vec![0]);
    writeln!(j, "  \"readme_pythagoras_3_4_5_proof\": \"{}\",", hex(&proof.dump_uncompressed())).unwrap();
    writeln!(j, "  \"readme_pythagoras_3_4_5_proof_compressed\": \"{}\",", hex(&proof.dump_compressed())).unwrap();
    assert!(circuit.verify(proof));
    let circuit = MulChain13::build();
    let proof = circuit.prove([3, 5], vec![0]);
    writeln!(j, "  \"mulchain_13_gates_proof\": \"{}\",", hex(&proof.dump_uncompressed())).unwrap();
    assert!(circuit.verify(proof));
    writeln!(j, "  \"fr_zero_is_zero\": {}", Fr::zero().is_zero()).unwrap();
    j.push_str("}\n");
    std::fs::write(&out_path, j).unwrap();
    eprintln!("wrote {}", out_path);
}
