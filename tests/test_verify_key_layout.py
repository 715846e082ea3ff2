"""CPU checks of the verification-key restatement (tests/verify_key_ref.py), which the GPU tests compare the library's
bytes with: the size formula, every field at its offset, and the sigma coefficients being the sigma columns of the
oracle's permutation."""
import pytest

from oracle.pyoracle import builder, kzg, poly, rng
from oracle.pyoracle.curve import G1_GEN, g1_deserialize_unchecked
from oracle.pyoracle.fields import R_MOD

import verify_key_ref as ref

TAU = rng.fr_rand_stream(1, 1)[0]


@pytest.fixture(scope="module")
def readme():
    oc = builder.compile_circuit(builder.circuit_pythagoras, 3, TAU)
    return oc, ref.vk_bytes_of(oc)


@pytest.mark.parametrize("n", [2, 8, 1024, 1 << 20])
def test_layout_offsets_and_size(n):
    off = ref.layout(n)
    assert off["size"] == 1376 + 64 * n
    assert off["g1"] == off["k"] + 3 * 32
    assert off["g2"] == off["g1"] + 9 * 96
    assert off["g2s"] == off["g2"] + 192
    assert off["sigma_1_len"] == off["g2s"] + 192
    assert off["sigma_2"] - off["sigma_2_len"] == 8


def test_fields_sit_at_their_offsets(readme):
    oc, raw = readme
    n = oc.domain.size
    off = ref.layout(n)
    assert len(raw) == off["size"]
    assert raw[:4] == b"TPVK" and int.from_bytes(raw[4:8], "little") == 1
    assert int.from_bytes(raw[8:16], "little") == n
    ks = [int.from_bytes(raw[off["k"] + 32 * i: off["k"] + 32 * i + 32], "little") for i in range(3)]
    assert ks == list(oc.copy_constrains.cosets)
    pts = [g1_deserialize_unchecked(raw[off["g1"] + 96 * i: off["g1"] + 96 * i + 96]) for i in range(9)]
    assert pts[:5] == list(oc.fixed_commitments)
    assert pts[8] == kzg.identity(oc.srs) == G1_GEN
    assert raw[off["g2"]: off["g2s"]] == ref.g2_wire(oc.srs.g2)
    assert raw[off["g2s"]: off["sigma_1_len"]] == ref.g2_wire(oc.srs.g2s)
    for s in (1, 2):
        assert int.from_bytes(raw[off["sigma_%d_len" % s]: off["sigma_%d_len" % s] + 8], "little") == n


def test_sigma_coefficients_are_the_permutation_columns(readme):
    oc, raw = readme
    n = oc.domain.size
    off = ref.layout(n)
    for s in range(2):
        at = off["sigma_%d" % (s + 1)]
        coef = [int.from_bytes(raw[at + 32 * i: at + 32 * i + 32], "little") for i in range(n)]
        assert all(c < R_MOD for c in coef)
        # evaluated over the domain: the sigma column of the compiled permutation (lib.rs:101-128)
        evals = oc.domain.fft(coef) if hasattr(oc.domain, "fft") else [poly.evaluate(coef, w) for w in oc.domain.elements()]
        assert evals == [cell[1] for cell in oc.copy_constrains.cols[s]]
    # the sigma commitments are commitments to these coefficients (and sigma_3's to the third column)
    sig = ref.sigma_coefficients(oc)
    pts = [g1_deserialize_unchecked(raw[off["g1"] + 96 * i: off["g1"] + 96 * i + 96]) for i in range(5, 8)]
    assert pts == [kzg.commit(oc.srs, poly.strip(c)) for c in sig]


def test_additive_and_chain_keys_have_the_formula_size():
    for run, inputs in ((builder.circuit_additive, 5), (builder.make_mul_chain(13), 2)):
        raw = ref.vk_bytes(run, inputs, TAU)
        n = int.from_bytes(raw[8:16], "little")
        assert n & (n - 1) == 0 and len(raw) == 1376 + 64 * n
