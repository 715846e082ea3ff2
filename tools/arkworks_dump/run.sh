#!/usr/bin/env bash
# usage: tools/arkworks_dump/run.sh /path/to/TyPLONK   (needs cargo + crates.io access)
# Copies the reference, makes its two sources of randomness deterministic (the ONLY change: tau and the nine blinders
# come from StdRng::seed_from_u64(1) / (2) instead of thread_rng -- the values bench.py and the tests use), runs the
# dumper and writes tests/golden/arkworks_vectors.json; tests/test_arkworks_vectors.py then stops skipping.
set -euo pipefail
here=$(cd "$(dirname "$0")" && pwd)
ref=${1:?path to a checkout of fabrizio-m/TyPLONK}
rm -rf "$here/ref" && mkdir -p "$here/ref"
cp -r "$ref/plonk" "$ref/kzg" "$ref/permutation" "$here/ref/"
# kzg/src/srs.rs:36-41  Srs::random: tau = Fr::rand(StdRng::seed_from_u64(1))
sed -i 's|let mut rng = rand::thread_rng();|let mut rng = <rand::rngs::StdRng as rand::SeedableRng>::seed_from_u64(1);|' "$here/ref/kzg/src/srs.rs"
# plonk/src/proof.rs:42  blinders = 9 x Fr::rand(StdRng::seed_from_u64(2)) in the order a0 a1 a2 b0 b1 b2 c0 c1 c2
sed -i 's|let mut rng = rand::thread_rng();|let mut rng = <rand::rngs::StdRng as rand::SeedableRng>::seed_from_u64(2);|' "$here/ref/plonk/src/proof.rs"
# the doc-test build script of the plonk crate is not needed here
sed -i '/^build = "build.rs"/d; /skeptic/d; /^\[build-dependencies\]/d; /^\[dev-dependencies\]/d' "$here/ref/plonk/Cargo.toml"
# an additive accessor (the fields of Proof are private): the proof as the concatenation of its items in declaration
# order (proof.rs:85-95), each in ark-serialize 0.3 uncompressed encoding -- the repository's canonical proof bytes
cat >> "$here/ref/plonk/src/proof.rs" <<'RS'

impl Proof {
    pub fn dump_uncompressed(&self) -> Vec<u8> {
        use ark_serialize::CanonicalSerialize;
        let mut v = vec![];
        for p in [&self.a, &self.b, &self.c] {
            p.commitment.0.serialize_unchecked(&mut v).unwrap();
            p.opening.0.serialize_unchecked(&mut v).unwrap();
            p.opening.1.serialize_uncompressed(&mut v).unwrap();
        }
        self.permutation.commitment.0.serialize_unchecked(&mut v).unwrap();
        self.permutation.z.0.serialize_unchecked(&mut v).unwrap();
        self.permutation.z.1.serialize_uncompressed(&mut v).unwrap();
        self.permutation.zw.0.serialize_unchecked(&mut v).unwrap();
        self.permutation.zw.1.serialize_uncompressed(&mut v).unwrap();
        self.evaluation_point.serialize_uncompressed(&mut v).unwrap();
        for t in self.t.iter() {
            t.0.serialize_unchecked(&mut v).unwrap();
        }
        self.r.0.serialize_unchecked(&mut v).unwrap();
        self.r.1.serialize_uncompressed(&mut v).unwrap();
        self.public_inputs.serialize_uncompressed(&mut v).unwrap();
        v
    }
    // the same items with `serialize`: compressed points (x and the y-sign flag), scalars unchanged
    pub fn dump_compressed(&self) -> Vec<u8> {
        use ark_serialize::CanonicalSerialize;
        let mut v = vec![];
        for p in [&self.a, &self.b, &self.c] {
            p.commitment.0.serialize(&mut v).unwrap();
            p.opening.0.serialize(&mut v).unwrap();
            p.opening.1.serialize(&mut v).unwrap();
        }
        self.permutation.commitment.0.serialize(&mut v).unwrap();
        self.permutation.z.0.serialize(&mut v).unwrap();
        self.permutation.z.1.serialize(&mut v).unwrap();
        self.permutation.zw.0.serialize(&mut v).unwrap();
        self.permutation.zw.1.serialize(&mut v).unwrap();
        self.evaluation_point.serialize(&mut v).unwrap();
        for t in self.t.iter() {
            t.0.serialize(&mut v).unwrap();
        }
        self.r.0.serialize(&mut v).unwrap();
        self.r.1.serialize(&mut v).unwrap();
        self.public_inputs.serialize(&mut v).unwrap();
        v
    }
}
RS
grep -q 'seed_from_u64(1)' "$here/ref/kzg/src/srs.rs" && grep -q 'seed_from_u64(2)' "$here/ref/plonk/src/proof.rs"
(cd "$here" && cargo run --release -- "$here/../../tests/golden/arkworks_vectors.json")
