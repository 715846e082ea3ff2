"""CPU: the MSM's lazy XYZZ addition laws (typlonk_b200/csrc/ec.cuh, FqOps<true>) restated operation by operation on
the generator's simulator of the very PTX forms the device runs (tools/gen_mont.py: products without their final
subtraction, sums / differences modulo 2q, the negations 1q - a and 2q - a, the normalisation to [0, q)).  Every
intermediate must stay below 2q -- the simulator's carry asserts check each form's internal bounds on the way -- and
the normalised results must be the points the oracle's big-integer G1 arithmetic gives, for generic sums, doubling
(P + P), cancellation (P + (-P)) and the identity, with bucket coordinates held non-canonically (x + q) and with
zeros mod q held as q."""
import os
import random
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_mont as G  # noqa: E402
from oracle.pyoracle import curve  # noqa: E402

Q = G.Q_MOD
N = 12
R = 1 << 384
RINV = pow(R, -1, Q)


class Lazy:
    """The device forms of field.cuh's lazy section, run on the simulator; every output is checked to be below 2q."""

    def __init__(self):
        self.mul_pr = G.build_mul(Q, N, reduce_final=False)
        self.mul2_pr = G.build_mul(Q, N, reduce_final=False, pair2=True)
        self.sqr_pr = G.build_sep(Q, N, "sqr", reduce_final=False)
        self.add_pr = G.build_add(2 * Q, N)
        self.sub_pr = G.build_sub(2 * Q, N)
        self.neg1_pr = G.build_kq_minus(Q, N, 1)
        self.neg2_pr = G.build_kq_minus(Q, N, 2)
        self.norm_pr = G.build_condsub(Q, N, (1,))
        self.ops = 0

    def _run(self, pr, bound=2 * Q, **vals):
        env = {}
        for nm, v in vals.items():
            assert 0 <= v <= 2 * Q, (nm, hex(v))
            for i, limb in enumerate(G.limbs(v, N)):
                env["%s%d" % (nm, i)] = limb
        out = pr.run(env)
        r = sum(out["r%d" % i] << (32 * i) for i in range(N))
        assert r < bound, hex(r)
        self.ops += 1
        return r

    def mul(self, a, b):
        r = self._run(self.mul_pr, a=a, b=b)
        assert r % Q == a * b * RINV % Q
        return r

    def sqr(self, a):
        r = self._run(self.sqr_pr, a=a)
        assert r % Q == a * a * RINV % Q
        return r

    def mul_sub2(self, a, b, c, d):   # fq_mul_sub2_lazy: a b + c (2q - d), one reduction
        nd = self._run(self.neg2_pr, bound=2 * Q + 1, a=d)
        r = self._run(self.mul2_pr, a=a, b=b, c=c, d=nd)
        assert r % Q == (a * b - c * d) * RINV % Q
        return r

    def add(self, a, b):
        return self._run(self.add_pr, a=a, b=b)

    def sub(self, a, b):
        return self._run(self.sub_pr, a=a, b=b)

    def dbl(self, a):
        return self.add(a, a)

    def neg(self, a):                 # fq_neg_lazy: a canonical, q - a in [1, q]
        assert a < Q
        return self._run(self.neg1_pr, bound=Q + 1, a=a)

    def norm(self, a):
        r = self._run(self.norm_pr, bound=Q, a=a)
        assert r == a % Q
        return r

    @staticmethod
    def is_zero(a):                   # fq_is_zero2: low-limb filter, then the full compare against 0 and q
        assert a < 2 * Q
        if (a & 0xFFFFFFFF) not in (0, Q & 0xFFFFFFFF):
            assert a % Q != 0
            return False
        return a in (0, Q)


F = Lazy()
ONE = R % Q


def identity():
    return [0, 0, 0, 0]


def is_identity(p):
    return p[2] == 0


def xyzz_mdbl(p):
    x, y = p
    u = F.dbl(y)
    v = F.sqr(u)
    w = F.mul(u, v)
    s = F.mul(x, v)
    xx = F.sqr(x)
    m = F.add(F.dbl(xx), xx)
    x3 = F.sub(F.sqr(m), F.dbl(s))
    y3 = F.mul_sub2(m, F.sub(s, x3), w, y)
    return [x3, y3, v, w]


def xyzz_dbl(r):
    if is_identity(r):
        return r
    x, y, zz, zzz = r
    u = F.dbl(y)
    v = F.sqr(u)
    w = F.mul(u, v)
    s = F.mul(x, v)
    xx = F.sqr(x)
    m = F.add(F.dbl(xx), xx)
    x3 = F.sub(F.sqr(m), F.dbl(s))
    y3 = F.mul_sub2(m, F.sub(s, x3), w, y)
    return [x3, y3, F.mul(v, zz), F.mul(w, zzz)]


def xyzz_madd(acc, p, neg):
    px, py = p
    if neg:
        py = F.neg(py)
    if is_identity(acc):
        return [px, py, ONE, ONE]
    x1, y1, zz1, zzz1 = acc
    u2 = F.mul(px, zz1)
    s2 = F.mul(py, zzz1)
    pp_ = F.sub(u2, x1)
    rr = F.sub(s2, y1)
    if F.is_zero(pp_):
        return xyzz_mdbl((px, py)) if F.is_zero(rr) else identity()
    pp = F.sqr(pp_)
    ppp = F.mul(pp_, pp)
    q = F.mul(x1, pp)
    x3 = F.sub(F.sub(F.sqr(rr), ppp), F.dbl(q))
    y3 = F.mul_sub2(rr, F.sub(q, x3), y1, ppp)
    return [x3, y3, F.mul(zz1, pp), F.mul(zzz1, ppp)]


def xyzz_add(acc, b):
    if is_identity(b):
        return acc
    if is_identity(acc):
        return list(b)
    x1, y1, zz1, zzz1 = acc
    x2, y2, zz2, zzz2 = b
    u1 = F.mul(x1, zz2)
    u2 = F.mul(x2, zz1)
    s1 = F.mul(y1, zzz2)
    s2 = F.mul(y2, zzz1)
    pp_ = F.sub(u2, u1)
    rr = F.sub(s2, s1)
    if F.is_zero(pp_):
        return xyzz_dbl(acc) if F.is_zero(rr) else identity()
    pp = F.sqr(pp_)
    ppp = F.mul(pp_, pp)
    q = F.mul(u1, pp)
    x3 = F.sub(F.sub(F.sqr(rr), ppp), F.dbl(q))
    y3 = F.mul_sub2(rr, F.sub(q, x3), s1, ppp)
    return [x3, y3, F.mul(F.mul(zz1, zz2), pp), F.mul(F.mul(zzz1, zzz2), ppp)]


# ---- conversions ---------------------------------------------------------------------------------------------------
def mont(x):
    return x * R % Q


def to_affine(p):
    """normalise (the device's last step), leave Montgomery form, divide out ZZ / ZZZ"""
    x, y, zz, zzz = (F.norm(c) * RINV % Q for c in p)
    if zz == 0:
        return None
    return x * pow(zz, -1, Q) % Q, y * pow(zzz, -1, Q) % Q


def table_point(pt):
    """a base as the MSM's tables hold it: canonical Montgomery coordinates"""
    return mont(pt[0]), mont(pt[1])


def scaled(pt, lam, rnd):
    """XYZZ form of an affine point with ZZ = lam^2, ZZZ = lam^3, every coordinate below q held as itself or + q"""
    x, y = pt
    c = [x * lam * lam % Q, y * lam ** 3 % Q, lam * lam % Q, lam ** 3 % Q]
    return [v + Q if rnd.random() < 0.5 else v for v in (mont(v) for v in c)]


def points(k, seed):
    rnd = random.Random(seed)
    return [curve.g1_mul(curve.G1_GEN, rnd.randrange(1, curve.R_MOD)) for _ in range(k)]


# ---- tests ---------------------------------------------------------------------------------------------------------
def test_mixed_addition_matches_oracle():
    pts = points(12, 1)
    acc = identity()
    want = None
    for i, p in enumerate(pts):
        neg = i % 3 == 2
        acc = xyzz_madd(acc, table_point(p), neg)
        want = curve.g1_add(want, curve.g1_neg(p) if neg else p)
        assert to_affine(acc) == want


def test_mixed_addition_doubling_and_cancellation():
    p, q = points(2, 2)
    tp = table_point(p)
    acc = xyzz_madd(identity(), tp, False)
    assert to_affine(xyzz_madd(acc, tp, False)) == curve.g1_add(p, p)        # P + P: the doubling branch
    assert is_identity(xyzz_madd(acc, tp, True))                              # P + (-P): the identity
    # the same with a bucket that reached P through other points (ZZ != 1, coordinates non-canonical)
    rnd = random.Random(3)
    acc = scaled(p, rnd.randrange(2, Q), rnd)
    assert to_affine(xyzz_madd(acc, tp, False)) == curve.g1_add(p, p)
    assert is_identity(xyzz_madd(acc, tp, True))
    acc = scaled(curve.g1_neg(q), rnd.randrange(2, Q), rnd)
    assert is_identity(xyzz_madd(acc, table_point(q), False))
    assert to_affine(xyzz_madd(acc, table_point(q), True)) == curve.g1_add(curve.g1_neg(q), curve.g1_neg(q))


def test_general_addition_matches_oracle():
    rnd = random.Random(4)
    pts = points(10, 5)
    for i in range(0, len(pts), 2):
        a, b = pts[i], pts[i + 1]
        for _ in range(3):
            pa = scaled(a, rnd.randrange(1, Q), rnd)
            pb = scaled(b, rnd.randrange(1, Q), rnd)
            assert to_affine(xyzz_add(pa, pb)) == curve.g1_add(a, b)
            assert to_affine(xyzz_add(pa, scaled(a, rnd.randrange(1, Q), rnd))) == curve.g1_add(a, a)   # doubling
            assert is_identity(xyzz_add(pa, scaled(curve.g1_neg(a), rnd.randrange(1, Q), rnd)))          # cancellation
            assert xyzz_add(pa, identity()) == pa and xyzz_add(identity(), pb) == pb


def test_running_sums_stay_bounded():
    """the reduction's running sums: long chains of general additions on lazy outputs (never re-normalised)"""
    rnd = random.Random(6)
    pts = points(16, 7)
    running, tot = identity(), identity()
    want_r, want_t = None, None
    for p in reversed(pts):
        running = xyzz_add(running, scaled(p, rnd.randrange(1, Q), rnd))
        tot = xyzz_add(tot, running)
        want_r = curve.g1_add(want_r, p)
        want_t = curve.g1_add(want_t, want_r)
    assert to_affine(running) == want_r
    assert to_affine(tot) == want_t
    doubled = xyzz_dbl(running)
    assert to_affine(doubled) == curve.g1_add(want_r, want_r)


def test_zero_tests_are_exact_on_lazy_values():
    """differences that are 0 mod q come out as 0 or q; both must read as zero, nothing else may"""
    assert Lazy.is_zero(0) and Lazy.is_zero(Q)
    for v in (1, Q - 1, Q + 1, 2 * Q - 1, (Q & 0xFFFFFFFF), Q + (1 << 32)):
        assert not Lazy.is_zero(v)
    x = mont(12345)
    assert F.sub(x, x) == 0
    assert F.sub(x + Q, x) in (0, Q) and F.sub(x, x + Q) in (0, Q)
    assert Lazy.is_zero(F.sub(x + Q, x)) and Lazy.is_zero(F.sub(x, x + Q))


@pytest.mark.parametrize("held", ["canonical", "plus_q"])
def test_worst_case_operands(held):
    """every bucket coordinate at the top of its range (values just below 2q, zeros mod q held as q) still gives bounded
    intermediates -- the laws' only inputs are < 2q values and canonical table points"""
    rnd = random.Random(8)
    p, b = points(2, 9)
    acc = scaled(p, rnd.randrange(1, Q), rnd)
    if held == "plus_q":
        acc = [v if v >= Q else v + Q for v in acc]
    else:
        acc = [v % Q for v in acc]
    worst_table = (Q - 1, Q - 1)   # not a curve point: only the bounds are checked here
    xyzz_madd(list(acc), worst_table, False)
    xyzz_madd(list(acc), worst_table, True)
    xyzz_add(list(acc), [2 * Q - 1] * 4)
    xyzz_dbl([2 * Q - 1, 2 * Q - 1, 2 * Q - 1, 2 * Q - 1])
    xyzz_mdbl((Q - 1, Q))
    assert to_affine(xyzz_madd(list(acc), table_point(b), False)) == curve.g1_add(p, b)
