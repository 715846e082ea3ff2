"""GPU tests of the SRS ceremony (csrc/srs_ceremony.cu, k_srs_contribute in csrc/srs.cu): a contribution equals the
SRS of the product secret byte for byte, on arbitrary bases too; the rebuilt tables commit and prove like a fresh SRS;
tp_srs_verify accepts powers and rejects every kind of damage; the link check; device groups; the C++ mirror."""
import os
import random
import subprocess

import pytest

from oracle.pyoracle import curve, fields, rng
from typlonk_b200 import ffi, field as F, synthetic
from typlonk_b200.ffi import Context
from typlonk_b200.kzg import KzgScheme, Srs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q, R = fields.Q_MOD, fields.R_MOD
TAU = rng.fr_rand_stream(1, 1)[0]
S1 = rng.fr_rand_stream(11, 1)[0]
S2 = rng.fr_rand_stream(12, 1)[0]


def _g2(pt):
    """oracle G2 point -> the g2_ref() shape"""
    return None if pt is None else ((pt[0].a, pt[0].b), (pt[1].a, pt[1].b))


def _off_subgroup_point():
    x = 0
    while True:
        x += 1
        rhs = (x ** 3 + 4) % Q
        y = pow(rhs, (Q + 1) // 4, Q)
        if y * y % Q == rhs and curve.g1_mul((x, y), R - 1) != curve.g1_neg((x, y)):
            return (x, y)


def _upload(ctx, points, g2=curve.G2_GEN, g2s=None):
    """an SRS from packed records (bytes) or oracle points, with the G2 points of TAU unless given"""
    raw = points if isinstance(points, (bytes, bytearray)) else b"".join(F.g1_to_packed(p) for p in points)
    srs = Srs(ctx, ctx.srs_upload(bytes(raw)))
    srs.handle.set_g2(F.g2_to_abi(_g2(g2)), F.g2_to_abi(_g2(curve.g2_mul(curve.G2_GEN, TAU) if g2s is None else g2s)))
    return srs


@pytest.mark.parametrize("gates", [5, (1 << 10) - 3, (1 << 16) + 1, (1 << 20) - 3])
def test_contribution_equals_the_srs_of_the_product_secret(ctx, gates):
    base = Srs.from_secret(ctx, TAU, gates)
    nxt, pub = base.contribute(S1)
    want = Srs.from_secret(ctx, TAU * S1 % R, gates)
    assert len(nxt) == gates + 3
    assert nxt.handle.download() == want.handle.download()
    assert nxt.handle.g2() == want.handle.g2()
    assert pub == _g2(curve.g2_mul(curve.G2_GEN, S1))
    assert base.handle.download(0, 4) == Srs.from_secret(ctx, TAU, 1).handle.download()   # the input is untouched
    if gates < (1 << 20):
        again, _ = nxt.contribute(S2)
        twice = Srs.from_secret(ctx, TAU * S1 * S2 % R, gates)
        assert again.handle.download() == twice.handle.download()
        assert again.handle.g2() == twice.handle.g2()
        for s in (again, twice):
            s.handle.destroy()
    for s in (base, nxt, want):
        s.handle.destroy()


def test_contribution_over_arbitrary_bases(ctx):
    rnd = random.Random(5)
    pts = [curve.g1_mul(curve.G1_GEN, rnd.randrange(1, R)) for _ in range(37)]
    pts.insert(20, None)
    srs = _upload(ctx, pts)
    nxt, pub = srs.contribute(S1)
    got = nxt.g1_ref()
    assert got == [curve.g1_mul(p, pow(S1, i, R)) if p is not None else None for i, p in enumerate(pts)]
    assert nxt.handle.download(20, 1) == bytes(96)
    assert nxt.g2s_ref() == _g2(curve.g2_mul(curve.G2_GEN, TAU * S1))
    assert nxt.g2_ref() == srs.g2_ref()


def test_contributed_srs_commits_and_proves_like_a_fresh_one(ctx):
    n = 1 << 10
    srs, _ = Srs.from_secret(ctx, TAU, n).contribute(S1)
    fresh = Srs.from_secret(ctx, TAU * S1 % R, n)
    poly = rng.fr_rand_stream(21, n + 3)
    assert KzgScheme(srs).commit(poly) == KzgScheme(fresh).commit(poly)
    t = synthetic.mul_chain_trace(n - 3)
    sel_all = t.selectors()
    sel = [bytes(sel_all[k * n * 32:(k + 1) * n * 32]) for k in range(5)]
    perm = bytes(t.permutation())
    cols = [F.fr_vec_to_bytes(c) for c in synthetic.mul_chain_witness(n - 3, n)]
    proofs = []
    for s in (srs, fresh):
        handle, _ = ctx.circuit_compile(s.handle, sel, perm, n)
        proofs.append(handle.prove_inputs(cols, bytes(32)))
        assert handle.verify(proofs[-1], bytes(32))
        handle.destroy()
    assert proofs[0] == proofs[1]


@pytest.mark.parametrize("log_len", [10, 20])
def test_verify_accepts_powers(ctx, log_len):
    gates = (1 << log_len) - 3
    srs = Srs.from_secret(ctx, TAU, gates)
    assert srs.verify()
    nxt, _ = srs.contribute(S1)
    assert nxt.verify()
    for s in (srs, nxt):
        s.handle.destroy()


def test_verify_rejects_each_kind_of_damage(ctx):
    good = bytearray(Srs.from_secret(ctx, TAU, 61).handle.download())
    n = len(good) // 96
    assert _upload(ctx, good).verify()

    def rec(i):
        return slice(96 * i, 96 * (i + 1))

    def damaged(i, pt):
        bad = bytearray(good)
        bad[rec(i)] = F.g1_to_packed(pt)
        return bad

    pts = [F.g1_from_packed(bytes(good[rec(i)])) for i in range(n)]
    cases = {
        "g1[0] != G (every point times 3)": (b"".join(F.g1_to_packed(curve.g1_mul(p, 3)) for p in pts), {}),
        "a middle point replaced": (damaged(30, curve.g1_mul(curve.G1_GEN, 12345)), {}),
        "the last point changed": (damaged(n - 1, curve.g1_add(pts[n - 1], curve.G1_GEN)), {}),
        "g2s of another tau": (good, {"g2s": curve.g2_mul(curve.G2_GEN, TAU + 1)}),
        "a point outside G1": (damaged(17, _off_subgroup_point()), {}),
        "an infinity record": (damaged(9, None), {}),
        "g2 not the generator": (good, {"g2": curve.g2_mul(curve.G2_GEN, 2), "g2s": curve.g2_mul(curve.G2_GEN, 2 * TAU)}),
    }
    swapped = bytearray(good)
    swapped[rec(40)], swapped[rec(41)] = good[rec(41)], good[rec(40)]
    cases["two adjacent points swapped"] = (swapped, {})
    for name, (raw, g2) in cases.items():
        srs = _upload(ctx, raw, **g2)
        assert not srs.verify(), name
        srs.handle.destroy()
    # argument errors: no G2 points, fewer than two points
    bare = Srs(ctx, ctx.srs_upload(bytes(good)))
    with pytest.raises(ffi.TyplonkError) as e:
        bare.verify()
    assert e.value.code == 1
    with pytest.raises(ffi.TyplonkError) as e:
        bare.contribute(S1)
    assert e.value.code == 1
    with pytest.raises(ffi.TyplonkError) as e:
        _upload(ctx, good[:96]).verify()
    assert e.value.code == 1


def test_update_link_and_secret_arguments(ctx):
    prev = Srs.from_secret(ctx, TAU, 29)
    nxt, pub = prev.contribute(S1)
    assert nxt.verify_update(prev, pub)
    assert not nxt.verify_update(prev, _g2(curve.g2_mul(curve.G2_GEN, S2)))
    assert not prev.verify_update(nxt, pub)
    tau_g1 = [F.g1_to_abi(F.g1_from_packed(s.handle.download(1, 1))) for s in (prev, nxt)]
    assert ffi.srs_update_check(tau_g1[0], tau_g1[1], F.g2_to_abi(pub))
    for bad in (bytes(32), R.to_bytes(32, "little"), b"\xff" * 32):
        with pytest.raises(ffi.TyplonkError) as e:
            ctx.srs_contribute(prev.handle, bad)
        assert e.value.code == 1
    # secrets drawn by the library: the results verify, link, and differ
    a, pa = prev.contribute()
    b, pb = prev.contribute()
    assert a.verify() and b.verify()
    assert a.verify_update(prev, pa) and b.verify_update(prev, pb)
    assert a.handle.download(1, 1) != b.handle.download(1, 1) and pa != pb


def test_device_group_of_two_ranks_on_one_device():
    g = Context.multi([0, 0])
    single = Context(0)
    try:
        gates = 1000
        srs, pub = Srs.from_secret(g, TAU, gates).contribute(S1)
        want, want_pub = Srs.from_secret(single, TAU, gates).contribute(S1)
        assert pub == want_pub
        assert srs.handle.download() == want.handle.download()
        assert srs.handle.g2() == want.handle.g2()
        # the sharded MSM reads every rank's copy: a full-length commitment equal to the single device's
        poly = rng.fr_rand_stream(31, gates + 3)
        assert KzgScheme(srs).commit(poly) == KzgScheme(want).commit(poly)
        assert srs.verify()
        raw = bytearray(want.handle.download())
        raw[96 * 7:96 * 8], raw[96 * 8:96 * 9] = raw[96 * 8:96 * 9], raw[96 * 7:96 * 8]
        bad = _upload(g, raw, g2s=curve.g2_mul(curve.G2_GEN, TAU * S1))
        assert not bad.verify()
        bad.handle.destroy()
    finally:
        single.close()
        g.close()


def test_cpp_srs_ceremony(tmp_path):
    from typlonk_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "typlonk_b200", "lib")
    exe = str(tmp_path / "srs_ceremony_test")
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                          "-o", exe, os.path.join(ROOT, "tests", "cpp", "srs_ceremony_test.cpp"),
                          "-L" + libdir, "-ltyplonk_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    res = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "FAIL" not in res.stdout and "0 failures" in res.stdout, res.stdout + res.stderr
