#!/usr/bin/env python3
"""Generator + CPU simulator for the Montgomery field kernels' inline PTX.

Emits typlonk_b200/csrc/mont_gen.cuh: one `asm` block per operation (mul, sqr-as-mul,
add, sub) for Fr (8 x u32 limbs) and Fq (12 x u32 limbs) of BLS12-381, with the modulus
limbs as PTX immediates.  Each operation is first built as a small IR (list of PTX-like
instructions) which this script *simulates* on random and edge-case operands against
Python big-int arithmetic, so the carry chains are proven correct on the CPU before any
GPU time is spent.

Multiplication is an interleaved (CIOS-style) Montgomery product over two accumulator
arrays ("even"/"odd" columns) so that every 32x32->64 product is a mad.lo.cc/madc.hi.cc
pair on an aligned register pair -- the pattern ptxas fuses into IMAD.WIDE.U32(.X).

Usage: python tools/gen_mont.py [--check-only] [--out PATH]
"""
import random
import sys
from pathlib import Path

R_MOD = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
Q_MOD = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
MASK = 0xFFFFFFFF


def limbs(x, n):
    return [(x >> (32 * i)) & MASK for i in range(n)]


class Prog:
    """Tiny PTX subset.  Registers are strings; ints are immediates."""

    def __init__(self):
        self.ins = []
        self.temps = []

    def emit(self, op, dst, *src, drop_carry=False):
        self.ins.append((op, dst, src, drop_carry))

    # ---- simulation ---------------------------------------------------------
    def run(self, env):
        cc = 0
        pred = {}

        def val(s):
            return s if isinstance(s, int) else env[s]

        for op, dst, src, drop in self.ins:
            s = [val(x) for x in src if not (isinstance(x, str) and x.startswith("%p"))]
            if op == "mul.lo.u32":
                env[dst] = (s[0] * s[1]) & MASK
            elif op == "mul.hi.u32":
                env[dst] = (s[0] * s[1]) >> 32
            elif op in ("mad.lo.cc.u32", "madc.lo.cc.u32"):
                cin = cc if op.startswith("madc") else 0
                t = ((s[0] * s[1]) & MASK) + s[2] + cin
                env[dst] = t & MASK
                cc = t >> 32
                if drop:
                    assert cc == 0, "dropped carry must be zero"
            elif op in ("mad.hi.cc.u32", "madc.hi.cc.u32", "madc.hi.u32"):
                cin = cc if op.startswith("madc") else 0
                t = ((s[0] * s[1]) >> 32) + s[2] + cin
                env[dst] = t & MASK
                if ".cc" in op:
                    cc = t >> 32
                    if drop:
                        assert cc == 0, "dropped carry must be zero"
                else:
                    assert t >> 32 == 0, "carry out of non-.cc op must be zero"
            elif op in ("add.cc.u32", "addc.cc.u32", "addc.u32", "add.u32"):
                cin = cc if op.startswith("addc") else 0
                t = s[0] + s[1] + cin
                env[dst] = t & MASK
                if ".cc" in op:
                    cc = t >> 32
                    if drop:
                        assert cc == 0, "dropped carry must be zero"
                elif drop:
                    assert t >> 32 == 0, "carry out must be zero"
            elif op in ("sub.cc.u32", "subc.cc.u32", "subc.u32"):
                bin_ = cc if op.startswith("subc") else 0
                t = s[0] - s[1] - bin_
                env[dst] = t & MASK
                if ".cc" in op:
                    cc = 1 if t < 0 else 0
            elif op == "sub.u32":
                env[dst] = (s[0] - s[1]) & MASK
            elif op == "shf.l.wrap.b32":
                env[dst] = ((s[1] << (s[2] & 31)) | (s[0] >> (32 - (s[2] & 31)))) & MASK
            elif op == "shl.b32":
                env[dst] = (s[0] << s[1]) & MASK
            elif op == "assert0":
                assert s[0] == 0, "limb expected to be zero"
            elif op == "setp.ne.u32":
                pred[dst] = s[0] != s[1]
            elif op == "selp.u32":
                env[dst] = s[0] if pred[src[2]] else s[1]
            elif op == "and.b32":
                env[dst] = s[0] & s[1]
            elif op == "mov.u32":
                env[dst] = s[0]
            else:
                raise ValueError(op)
        return env

    # ---- PTX text -----------------------------------------------------------
    def text(self, regmap):
        def r(x):
            if isinstance(x, int):
                return "0x%08x" % x
            return regmap.get(x, x)

        lines = []
        for op, dst, src, _ in self.ins:
            if op == "assert0":
                continue
            lines.append("%s %s, %s;" % (op, r(dst), ", ".join(r(x) for x in src)))
        return lines


def cond_sub_p(pr, t, d, out, mod, n):
    """out = t >= p ? t - p : t   (t < 2p < 2^(32n))."""
    pl = limbs(mod, n)
    for i in range(n):
        pr.emit("sub.cc.u32" if i == 0 else "subc.cc.u32", d[i], t[i], pl[i])
    pr.emit("subc.u32", "brw", 0, 0)
    pr.emit("setp.ne.u32", "%pb", "brw", 0)
    for i in range(n):
        pr.emit("selp.u32", out[i], t[i], d[i], "%pb")


def build_mul(mod, n, reduce_final=True, mod_regs=False, m0_reg=False, special=False, pair2=False):
    """special=True replaces products by modulus limbs equal to 1 / 0xffffffff (Fr's two lowest
    limbs) with additions: 16 of the 128 products of an Fr multiplication."""
    pl = ["p%d" % i for i in range(n)] if mod_regs else limbs(mod, n)
    m0 = (-pow(mod, -1, 1 << 32)) & MASK
    if m0_reg:
        m0 = "m0"  # register operand, see main()
    pr = Prog()
    a = ["a%d" % i for i in range(n)]
    b = ["b%d" % i for i in range(n)]
    X = ["e%d" % i for i in range(n)]
    Y = ["o%d" % i for i in range(n)]
    c2 = ["c%d" % i for i in range(n)]
    d2 = ["d%d" % i for i in range(n)]

    def cmad(acc, src, off, m):
        """acc[j],acc[j+1] += src[j+off]*m for j = 0,2,..; leaves carry in CC."""
        for j in range(0, n, 2):
            lim = src[j + off]
            if special and lim == 1 and j == 0:
                # m * 1: no multiplier needed
                pr.emit("add.cc.u32", acc[j], acc[j], m)
                pr.emit("addc.cc.u32", acc[j + 1], acc[j + 1], 0)
                continue
            if special and lim == MASK and j == 0:
                # m * (2^32 - 1) = (hm : nm) with nm = -m, hm = m - (m != 0), prepared by the caller
                pr.emit("add.cc.u32", acc[j], acc[j], "nm")
                pr.emit("addc.cc.u32", acc[j + 1], acc[j + 1], "hm")
                continue
            pr.emit("mad.lo.cc.u32" if j == 0 else "madc.lo.cc.u32", acc[j], lim, m, acc[j])
            pr.emit("madc.hi.cc.u32", acc[j + 1], lim, m, acc[j + 1], drop_carry=(off == 1 and j == n - 2))

    def mad_n_redc(even, odd, bi, first, di=None):
        if first:
            for j in range(0, n, 2):
                pr.emit("mul.lo.u32", odd[j], a[j + 1], bi)
                pr.emit("mul.hi.u32", odd[j + 1], a[j + 1], bi)
            for j in range(0, n, 2):
                pr.emit("mul.lo.u32", even[j], a[j], bi)
                pr.emit("mul.hi.u32", even[j + 1], a[j], bi)
        else:
            pr.emit("add.cc.u32", even[0], even[0], odd[1])
            for j in range(0, n - 2, 2):
                pr.emit("madc.lo.cc.u32", odd[j], a[j + 1], bi, odd[j + 2])
                pr.emit("madc.hi.cc.u32", odd[j + 1], a[j + 1], bi, odd[j + 3])
            pr.emit("madc.lo.cc.u32", odd[n - 2], a[n - 1], bi, 0)
            pr.emit("madc.hi.u32", odd[n - 1], a[n - 1], bi, 0)
            cmad(even, a, 0, bi)
            pr.emit("addc.u32", odd[n - 1], odd[n - 1], 0, drop_carry=True)
        if di is not None:
            # lazy pair: a second product row c * d_i joins before the shared reduction row
            cmad(odd, c2, 1, di)
            cmad(even, c2, 0, di)
            pr.emit("addc.u32", odd[n - 1], odd[n - 1], 0, drop_carry=True)
        pr.emit("mul.lo.u32", "mi", even[0], m0)
        if special and pl[1] == MASK:
            pr.emit("sub.cc.u32", "nm", 0, "mi")   # borrow <=> mi != 0
            pr.emit("subc.u32", "hm", "mi", 0)
        cmad(odd, pl, 1, "mi")
        cmad(even, pl, 0, "mi")
        pr.emit("addc.u32", odd[n - 1], odd[n - 1], 0, drop_carry=True)

    for i in range(0, n, 2):
        mad_n_redc(X, Y, b[i], first=(i == 0), di=d2[i] if pair2 else None)
        mad_n_redc(Y, X, b[i + 1], first=False, di=d2[i + 1] if pair2 else None)
    # merge: X[i] += Y[i+1]
    pr.emit("add.cc.u32", X[0], X[0], Y[1])
    for i in range(1, n - 1):
        pr.emit("addc.cc.u32", X[i], X[i], Y[i + 1])
    pr.emit("addc.u32", X[n - 1], X[n - 1], 0, drop_carry=True)
    out = ["r%d" % i for i in range(n)]
    if reduce_final:
        cond_sub_p(pr, X, Y, out, mod, n)  # Y reused as scratch for t - p
    else:
        for i in range(n):
            pr.emit("mov.u32", out[i], X[i])
    return pr


def build_add(mod, n):
    pr = Prog()
    a = ["a%d" % i for i in range(n)]
    b = ["b%d" % i for i in range(n)]
    t = ["e%d" % i for i in range(n)]
    d = ["o%d" % i for i in range(n)]
    for i in range(n):
        op = "add.cc.u32" if i == 0 else ("addc.cc.u32" if i < n - 1 else "addc.u32")
        pr.emit(op, t[i], a[i], b[i], drop_carry=(i == n - 1))
    cond_sub_p(pr, t, d, ["r%d" % i for i in range(n)], mod, n)
    return pr


def build_sub(mod, n):
    pl = limbs(mod, n)
    pr = Prog()
    a = ["a%d" % i for i in range(n)]
    b = ["b%d" % i for i in range(n)]
    t = ["e%d" % i for i in range(n)]
    for i in range(n):
        pr.emit("sub.cc.u32" if i == 0 else "subc.cc.u32", t[i], a[i], b[i])
    pr.emit("subc.u32", "brw", 0, 0)  # 0xffffffff on borrow
    for i in range(n):
        pr.emit("and.b32", "o%d" % i, "brw", pl[i])
    for i in range(n):
        op = "add.cc.u32" if i == 0 else ("addc.cc.u32" if i < n - 1 else "addc.u32")
        pr.emit(op, "r%d" % i, t[i], "o%d" % i)
    return pr


# ---- lazy Fr arithmetic for the NTT butterflies: values stay in [0, 2r) -----------------------------------------------
# r = 0.905 * 2^255, so 2r < 2^256 (and 4r is not: Harvey's [0, 4p) butterfly does not fit).  A Montgomery product of
# x < 2r by a reduced twiddle w < r is (x w + m r) / R < r (2r / R + 1) < 2r WITHOUT the final conditional subtraction,
# and sums / differences are reduced modulo 2r instead of r: the product's subtraction is what a butterfly saves; the
# transform's last store brings the values back to [0, r).
def build_add2(mod, n):
    """r = a + b reduced once by 2p; a, b < 2p, 2p < 2^(32 n) <= 4p possible: the sum may carry out of n limbs"""
    m2 = limbs(2 * mod, n)
    pr = Prog()
    a = ["a%d" % i for i in range(n)]
    b = ["b%d" % i for i in range(n)]
    t = ["e%d" % i for i in range(n)]
    d = ["o%d" % i for i in range(n)]
    for i in range(n):
        pr.emit("add.cc.u32" if i == 0 else "addc.cc.u32", t[i], a[i], b[i])
    pr.emit("addc.u32", "mi", 0, 0)                      # the carry: bit 32 n of the sum
    for i in range(n):
        pr.emit("sub.cc.u32" if i == 0 else "subc.cc.u32", d[i], t[i], m2[i])
    pr.emit("subc.u32", "brw", "mi", 0)                  # carry - borrow: non-zero exactly when the sum is below 2p
    pr.emit("setp.ne.u32", "%pb", "brw", 0)
    for i in range(n):
        pr.emit("selp.u32", "r%d" % i, t[i], d[i], "%pb")
    return pr


def build_condsub(mod, n, mults):
    """r = a reduced by one conditional subtraction of k p for every k in `mults`"""
    pr = Prog()
    # the selects below read their operand limb by limb while writing the result: work on a copy, the asm outputs are
    # not early-clobber and may share registers with the inputs (ptxas folds the moves away)
    cur = ["c%d" % i for i in range(n)]
    pr.temps = list(cur) + ["d%d" % i for i in range(n)]
    for i in range(n):
        pr.emit("mov.u32", cur[i], "a%d" % i)
    for step, k in enumerate(mults):
        last = step == len(mults) - 1
        out = ["r%d" % i for i in range(n)] if last else ["d%d" % i for i in range(n)]
        cond_sub_p(pr, cur, ["o%d" % i for i in range(n)], out, k * mod, n)
        cur = out
    return pr


def check_lazy(mod, n, trials=3000):
    R = 1 << (32 * n)
    assert 2 * mod < R
    rinv = pow(R, -1, mod)
    rnd = random.Random(4242)
    mul = build_mul(mod, n, reduce_final=False, m0_reg=True, special=True)
    mulfull = build_mul(mod, n, m0_reg=True, special=True)
    add2 = build_add2(mod, n)
    sub2 = build_sub(2 * mod, n)
    norm2 = build_condsub(mod, n, (1,))

    def run(pr, **vals):
        env = {"m0": (-pow(mod, -1, 1 << 32)) & MASK}
        for nm, v in vals.items():
            for i, l in enumerate(limbs(v, n)):
                env["%s%d" % (nm, i)] = l
        o = pr.run(env)
        return sum(o["r%d" % i] << (32 * i) for i in range(n))

    big = [0, 1, mod - 1, mod, mod + 1, 2 * mod - 2, 2 * mod - 1, R - 2 * mod, (R - 1) % (2 * mod),
           (1 << 255) - 1, 1 << 255, (1 << 255) + 1]
    small = [0, 1, 2, mod - 1, mod - 2, (mod - 1) // 2, R % mod]
    cases = [(x, w) for x in big for w in small] + [(rnd.randrange(2 * mod), rnd.randrange(mod)) for _ in range(trials)]
    for x, w in cases:
        # The reduced operand goes FIRST: it is the one whose limbs form the rows' multiplicand, and the interleaved
        # form's no-carry shortcut needs that one below 2^255; the second operand's limbs are only row multipliers and
        # may be anything below 2^256 (the other order fails the simulator's carry asserts, as it should).
        t = run(mul, a=w, b=x)
        assert t < 2 * mod and t % mod == x * w * rinv % mod, ("lazy mul", hex(x), hex(w))
        # the full product (last store of an inverse transform) takes a lazy operand and returns a canonical value
        assert run(mulfull, a=w, b=x) == x * w * rinv % mod
    cases = [(u, t) for u in big for t in big] + [(rnd.randrange(2 * mod), rnd.randrange(2 * mod)) for _ in range(trials)]
    for u, t in cases:
        s = run(add2, a=u, b=t)
        d = run(sub2, a=u, b=t)
        assert s < 2 * mod and s % mod == (u + t) % mod, ("add2", hex(u), hex(t))
        assert d < 2 * mod and d % mod == (u - t) % mod, ("sub2", hex(u), hex(t))
    for u in big + [rnd.randrange(2 * mod) for _ in range(trials)]:
        assert run(norm2, a=u) == u % mod
    print("%d-limb lazy forms ok" % n)


# ---- lazy Fq arithmetic for the MSM's XYZZ addition laws: values stay in [0, 2q) ---------------------------------------
# q = 0.8126 * 2^381, so 8q < R = 2^384.  A Montgomery product (a b + m q) / R of a, b < 2q is below q (4q / R + 1) <
# 1.41 q, and a lazy pair a b + c d of operands <= 2q (8 q^2 < q R) below q (8q / R + 1) < 1.82 q: none of the products
# needs its final conditional subtraction.  Sums and differences are taken modulo 2q (the same cost as modulo q), so
# every value between a table load and the last store of the reduction lies in [0, 2q); fq_norm2 returns to [0, q).
# Unreduced sums or differences (up to 4q) would save the correction of a sum or difference too, but a square of such
# a value is only bounded by q (16q / R + 1) > 2q: the laws square their differences (PP = (U2 - X1)^2, R^2).
def build_kq_minus(mod, n, k):
    """r = k p - a for a <= k p (no correction): a negation into [0, k p]"""
    kl = limbs(k * mod, n)
    pr = Prog()
    for i in range(n):
        op = "sub.cc.u32" if i == 0 else ("subc.cc.u32" if i < n - 1 else "subc.u32")
        pr.emit(op, "r%d" % i, kl[i], "a%d" % i)
    return pr


def check_lazy_fq(mod, n, trials=2000):
    R = 1 << (32 * n)
    assert 8 * mod < R
    rinv = pow(R, -1, mod)
    rnd = random.Random(4243)
    uid = _uid[0]   # the emitted header's temporary names stay what they were before this check existed
    mul = build_mul(mod, n, reduce_final=False)
    mul2 = build_mul(mod, n, reduce_final=False, pair2=True)
    sqr = build_sep(mod, n, "sqr", reduce_final=False)
    _uid[0] = uid
    add2 = build_add(2 * mod, n)
    sub2 = build_sub(2 * mod, n)
    neg1 = build_kq_minus(mod, n, 1)
    neg2 = build_kq_minus(mod, n, 2)
    norm2 = build_condsub(mod, n, (1,))

    def run(pr, **vals):
        env = {}
        for nm, v in vals.items():
            for i, l in enumerate(limbs(v, n)):
                env["%s%d" % (nm, i)] = l
        o = pr.run(env)
        return sum(o["r%d" % i] << (32 * i) for i in range(n))

    # edge operands of the lazy range [0, 2q): values = 0 mod q held as 0 and q, the ends of both halves, all-ones limbs
    big = [0, 1, mod - 1, mod, mod + 1, 2 * mod - 2, 2 * mod - 1, (1 << 381) - 1, 1 << 380, (R - 1) % (2 * mod),
           ((1 << (16 * n)) - 1) % (2 * mod), mod // 2, R % mod]
    lazy = big + [rnd.randrange(2 * mod) for _ in range(trials)]
    cases = [(x, y) for x in big for y in big] + [(rnd.randrange(2 * mod), rnd.randrange(2 * mod)) for _ in range(trials)]
    for x, y in cases:
        # both operand orders: the interleaved form's carry asserts accept any pair below 2q
        for a, b in ((x, y), (y, x)):
            t = run(mul, a=a, b=b)
            assert t < 2 * mod and t % mod == a * b * rinv % mod, ("lazy mul", hex(a), hex(b))
        t = run(sqr, a=x)
        assert t < 2 * mod and t % mod == x * x * rinv % mod, ("lazy sqr", hex(x))
        s = run(add2, a=x, b=y)
        d = run(sub2, a=x, b=y)
        assert s < 2 * mod and s % mod == (x + y) % mod, ("add2", hex(x), hex(y))
        assert d < 2 * mod and d % mod == (x - y) % mod, ("sub2", hex(x), hex(y))
    # lazy pair: a b + c (2q - d), the subtrahend's negation (0, 2q] included
    quads = [(x, y, c, d) for x in big[:8] for y in big[:8] for c in big[:8] for d in big[:8]]
    quads += [tuple(rnd.randrange(2 * mod) for _ in range(4)) for _ in range(trials)]
    for x, y, c, d in quads:
        nd = run(neg2, a=d)
        assert nd == 2 * mod - d
        t = run(mul2, a=x, b=y, c=c, d=nd)
        assert t < 2 * mod and t % mod == (x * y - c * d) * rinv % mod, ("lazy pair", hex(x), hex(y), hex(c), hex(d))
    for u in lazy:
        assert run(norm2, a=u) == u % mod
    for u in [0, 1, mod - 1] + [rnd.randrange(mod) for _ in range(trials)]:
        assert run(neg1, a=u) == mod - u
    print("%d-limb lazy Fq forms ok" % n)


# appended section for tools/gen_mont.py: separated-form (wide product + reduction) builders
class Cols:
    """Column accumulators in two alignments over absolute limb positions: E holds 64-bit pairs at
    (even, even+1), O at (odd, odd+1), so that every 32x32->64 product is a mad.lo.cc/madc.hi.cc
    pair on an aligned register pair whatever the parity of its position.  `fresh` limbs hold no
    value yet (they read as 0 and cost no instruction to initialise); `small` limbs hold <= 2."""

    def __init__(self, pr, prefix, size):
        self.pr = pr
        self.size = size
        self.reg = {0: ["%se%d" % (prefix, k) for k in range(size)],
                    1: ["%so%d" % (prefix, k) for k in range(size)]}
        self.fresh = {0: [True] * size, 1: [True] * size}
        self.small = {0: [False] * size, 1: [False] * size}

    def regs(self):
        return self.reg[0] + self.reg[1]

    def load(self, par, pos, src):
        """alias-free initialisation: limb `pos` of alignment `par` := register src"""
        self.pr.emit("mov.u32", self.reg[par][pos], src)
        self.fresh[par][pos] = False

    def chain(self, terms, carry_in=False):
        """terms: [(pos, x, y)] with pos rising by 2; all on the alignment pos & 1."""
        pr = self.pr
        par = terms[0][0] & 1
        reg, fresh, small = self.reg[par], self.fresh[par], self.small[par]
        use_c = carry_in
        for t, (pos, x, y) in enumerate(terms):
            assert (pos & 1) == par and (t == 0 or pos == terms[t - 1][0] + 2)
            last = t == len(terms) - 1
            lo_add = 0 if fresh[pos] else reg[pos]
            hi_add = 0 if fresh[pos + 1] else reg[pos + 1]
            if fresh[pos] and fresh[pos + 1] and not use_c:
                pr.emit("mul.lo.u32", reg[pos], x, y)
                pr.emit("mul.hi.u32", reg[pos + 1], x, y)
                fresh[pos] = fresh[pos + 1] = False
                use_c = False
                continue
            pr.emit("madc.lo.cc.u32" if use_c else "mad.lo.cc.u32", reg[pos], x, y, lo_add)
            hi_fresh = fresh[pos + 1]
            fresh[pos] = False
            small[pos] = False
            fresh[pos + 1] = False
            small[pos + 1] = False
            if hi_fresh:
                # hi + 0 + carry cannot overflow: the chain's carry ends here
                pr.emit("madc.hi.u32", reg[pos + 1], x, y, 0)
                use_c = False
                continue
            pr.emit("madc.hi.cc.u32", reg[pos + 1], x, y, hi_add)
            use_c = True
            if last:
                p = pos + 2
                while True:
                    if p >= self.size:
                        # top of the array: the value is known to fit
                        self.pr.ins[-1] = self.pr.ins[-1][:3] + (True,)
                        break
                    if fresh[p]:
                        pr.emit("addc.u32", reg[p], 0, 0)
                        fresh[p] = False
                        small[p] = True
                        break
                    if small[p]:
                        pr.emit("addc.u32", reg[p], reg[p], 0, drop_carry=True)
                        break
                    pr.emit("addc.cc.u32", reg[p], reg[p], 0)
                    p += 1

    def merge(self, lo, hi, out):
        """out[k - lo] = E[k] + O[k] for k in [lo, hi) with carries; the carry out of the top is dropped
        (checked by the simulator)."""
        pr = self.pr
        started = False
        for k in range(lo, hi):
            e = None if self.fresh[0][k] else self.reg[0][k]
            o = None if self.fresh[1][k] else self.reg[1][k]
            dst = out[k - lo]
            top = k == hi - 1
            if e is None and o is None:
                if started:
                    pr.emit("addc.cc.u32" if not top else "addc.u32", dst, 0, 0, drop_carry=top)
                else:
                    pr.emit("mov.u32", dst, 0)
                continue
            if e is None or o is None:
                src = e if o is None else o
                if started:
                    pr.emit("addc.cc.u32" if not top else "addc.u32", dst, src, 0, drop_carry=top)
                else:
                    pr.emit("mov.u32", dst, src)
                continue
            if not started:
                pr.emit("add.cc.u32" if not top else "add.u32", dst, e, o, drop_carry=top)
                started = True
            else:
                pr.emit("addc.cc.u32" if not top else "addc.u32", dst, e, o, drop_carry=top)


def wide_schoolbook(pr, cols, a, b, base=0):
    """cols += a * b << (32 base)  (rows of b; two chains per row)."""
    na, nb = len(a), len(b)
    for i in range(nb):
        for par in (0, 1):
            terms = [(base + i + j, a[j], b[i]) for j in range(par, na, 2)]
            if terms:
                cols.chain(terms)


def wide_square_cross(pr, cols, a):
    """cols += sum_{i<j} a_i a_j 2^(32 (i+j))"""
    n = len(a)
    for i in range(n):
        for par in (0, 1):
            terms = [(i + j, a[j], a[i]) for j in range(i + 1, n) if (j - i) % 2 == par]
            # same parity of (i + j) within the list, positions rise by 2
            if terms:
                cols.chain(terms)


_uid = [0]


def fresh_names(prefix, n):
    _uid[0] += 1
    return ["%s%d_%d" % (prefix, _uid[0], k) for k in range(n)]


def emit_wide_mul(pr, a, b, t, temps, karatsuba=False):
    """t[0 .. len(a)+len(b)) = a * b as plain limbs."""
    n = len(a)
    if not karatsuba:
        _uid[0] += 1
        cols = Cols(pr, "w%d" % _uid[0], 2 * n + 1)
        temps += cols.regs()
        wide_schoolbook(pr, cols, a, b)
        cols.merge(0, 2 * n, t)
        return
    h = n // 2
    a0, a1, b0, b1 = a[:h], a[h:], b[:h], b[h:]
    z0 = t[:n]
    z2 = t[n:]
    emit_wide_mul(pr, a0, b0, z0, temps)
    emit_wide_mul(pr, a1, b1, z2, temps)
    sa = fresh_names("sa", h)
    sb = fresh_names("sb", h)
    ca, cb = fresh_names("ck", 2)
    temps += sa + sb + [ca, cb]
    for (s, x0, x1, c) in ((sa, a0, a1, ca), (sb, b0, b1, cb)):
        for k in range(h):
            pr.emit("add.cc.u32" if k == 0 else "addc.cc.u32", s[k], x0[k], x1[k])
        pr.emit("addc.u32", c, 0, 0)           # 0 / 1
    zm = fresh_names("zm", n + 1)
    temps += zm
    emit_wide_mul(pr, sa, sb, zm[:n], temps)
    # + (ca * sb + cb * sa) << (32 h) + (ca & cb) << (32 n)
    ma, mb = fresh_names("mk", 2)
    temps += [ma, mb]
    pr.emit("sub.u32", ma, 0, ca)                # all-ones mask when the carry bit is set
    pr.emit("sub.u32", mb, 0, cb)
    tmp = fresh_names("kt", h)
    temps += tmp
    pr.emit("and.b32", zm[n], ca, cb)
    for (mask, s) in ((ma, sb), (mb, sa)):
        for k in range(h):
            pr.emit("and.b32", tmp[k], s[k], mask)
        for k in range(h):
            pr.emit("add.cc.u32" if k == 0 else "addc.cc.u32", zm[h + k], zm[h + k], tmp[k])
        pr.emit("addc.u32", zm[n], zm[n], 0, drop_carry=True)
    # zm -= z0 + z2
    for z in (z0, z2):
        for k in range(n):
            pr.emit("sub.cc.u32" if k == 0 else "subc.cc.u32", zm[k], zm[k], z[k])
        pr.emit("subc.u32", zm[n], zm[n], 0)
    # t += zm << (32 h)
    for k in range(n + 1):
        pr.emit("add.cc.u32" if k == 0 else "addc.cc.u32", t[h + k], t[h + k], zm[k])
    for k in range(h + n + 1, 2 * n):
        last = k == 2 * n - 1
        pr.emit("addc.cc.u32" if not last else "addc.u32", t[k], t[k], 0, drop_carry=last)


def emit_wide_sqr(pr, a, t, temps):
    n = len(a)
    _uid[0] += 1
    cols = Cols(pr, "q%d" % _uid[0], 2 * n + 1)
    temps += cols.regs()
    wide_square_cross(pr, cols, a)
    c = fresh_names("cr", 2 * n)
    temps += c
    cols.merge(0, 2 * n, c)
    # double: t = c << 1
    for k in range(2 * n - 1, 0, -1):
        pr.emit("shf.l.wrap.b32", t[k], c[k - 1], c[k], 1)
    pr.emit("shl.b32", t[0], c[0], 1)
    # + squares on the diagonal: one carry chain of n wide multiply-adds
    for i in range(n):
        pr.emit("mad.lo.cc.u32" if i == 0 else "madc.lo.cc.u32", t[2 * i], a[i], a[i], t[2 * i])
        last = i == n - 1
        pr.emit("madc.hi.cc.u32" if not last else "madc.hi.u32", t[2 * i + 1], a[i], a[i], t[2 * i + 1],
                drop_carry=last)


def emit_redc(pr, t, out, mod, n, temps, m0=None, reduce_final=True):
    """out = t / 2^(32 n) mod p (conditionally subtracted once), t = 2n plain limbs, t < p * 2^(32 n)
    (or < 2 p^2 for a lazy pair -- the callers' bounds are checked by the simulator's carry asserts).
    reduce_final=False: out = (t + m p) / 2^(32 n) < 2 p, without the subtraction."""
    pl = limbs(mod, n)
    if m0 is None:
        m0 = (-pow(mod, -1, 1 << 32)) & MASK
    _uid[0] += 1
    w = Cols(pr, "r%d" % _uid[0], n + n + 2)
    temps += w.regs()
    mi = "mi"
    for k in range(n):
        w.reg[0][k] = t[k]          # the even-aligned window starts as the low half of t (clobbered)
        w.fresh[0][k] = False
    for i in range(n):
        par = i & 1
        cur, oth = w.reg[par][i], w.reg[1 - par][i]
        carry_in = False
        if not w.fresh[1 - par][i]:
            pr.emit("add.cc.u32", cur, cur, oth)
            carry_in = True
        pr.emit("mul.lo.u32", mi, cur, m0)
        # products that land on the other alignment (positions i + j with j odd) take the merge carry
        w.chain([(i + j, pl[j], mi) for j in range(1, n, 2)], carry_in=carry_in)
        w.chain([(i + j, pl[j], mi) for j in range(0, n, 2)])
    # result = window[n .. 2n) + t[n .. 2n)
    s = fresh_names("rs", n + 1)
    temps += s
    w.merge(n, 2 * n + 1, s)
    for k in range(n):
        pr.emit("add.cc.u32" if k == 0 else "addc.cc.u32", s[k], s[k], t[n + k])
    pr.emit("addc.u32", s[n], s[n], 0, drop_carry=True)
    # s < 2p (s[n] is zero whenever the inputs respect the bound; asserted through the cond-sub test)
    if not reduce_final:
        pr.emit("assert0", None, s[n])
        for i in range(n):
            pr.emit("mov.u32", out[i], s[i])
        return
    d = fresh_names("rd", n)
    temps += d
    cond_sub_p(pr, s[:n], d, out, mod, n)


def build_sep(mod, n, kind, karatsuba=False, reduce_final=True):
    """kind: 'mul' (a*b), 'sqr' (a*a), 'mul2' (a*b + c*d)"""
    pr = Prog()
    a = ["a%d" % i for i in range(n)]
    b = ["b%d" % i for i in range(n)]
    temps = []
    t = fresh_names("t", 2 * n)
    temps += t
    if kind == "mul":
        emit_wide_mul(pr, a, b, t, temps, karatsuba)
    elif kind == "sqr":
        emit_wide_sqr(pr, a, t, temps)
    elif kind == "mul2":
        c = ["c%d" % i for i in range(n)]
        d = ["d%d" % i for i in range(n)]
        emit_wide_mul(pr, a, b, t, temps, karatsuba)
        t2 = fresh_names("u", 2 * n)
        temps += t2
        emit_wide_mul(pr, c, d, t2, temps, karatsuba)
        for k in range(2 * n):
            last = k == 2 * n - 1
            pr.emit("add.cc.u32" if k == 0 else ("addc.cc.u32" if not last else "addc.u32"), t[k], t[k], t2[k],
                    drop_carry=last)
    out = ["r%d" % i for i in range(n)]
    emit_redc(pr, t, out, mod, n, temps, reduce_final=reduce_final)
    pr.temps = temps
    return pr


def check(name, mod, n, trials=300, mod_regs=False, m0_reg=False, special=False):
    R = 1 << (32 * n)
    rinv = pow(R, -1, mod)
    mul = build_mul(mod, n, mod_regs=mod_regs, m0_reg=m0_reg, special=special)
    add = build_add(mod, n)
    sub = build_sub(mod, n)
    rnd = random.Random(1234 + n)
    edge = [0, 1, 2, mod - 1, mod - 2, (mod - 1) // 2, R % mod, (1 << (32 * n - 1)) % mod]
    cases = [(x, y) for x in edge for y in edge]
    cases += [(rnd.randrange(mod), rnd.randrange(mod)) for _ in range(trials)]
    for x, y in cases:
        env = {}
        for i, v in enumerate(limbs(x, n)):
            env["a%d" % i] = v
        for i, v in enumerate(limbs(y, n)):
            env["b%d" % i] = v
        for i, v in enumerate(limbs(mod, n)):
            env["p%d" % i] = v
        env["m0"] = (-pow(mod, -1, 1 << 32)) & MASK
        out = mul.run(dict(env))
        got = sum(out["r%d" % i] << (32 * i) for i in range(n))
        assert got == x * y * rinv % mod, (name, "mul", hex(x), hex(y))
        out = add.run(dict(env))
        got = sum(out["r%d" % i] << (32 * i) for i in range(n))
        assert got == (x + y) % mod, (name, "add")
        out = sub.run(dict(env))
        got = sum(out["r%d" % i] << (32 * i) for i in range(n))
        assert got == (x - y) % mod, (name, "sub")
    nmad = sum(1 for i in mul.ins if i[0].startswith(("mad", "mul")))
    print("%s: %d cases ok; mul = %d PTX instrs (%d mul/mad)" % (name, len(cases), len(mul.ins), nmad))


def emit_fn(fname, pr, n, mod_sym=None, m0_sym=None):
    regmap = {}
    if m0_sym:
        regmap["m0"] = "%%%d" % (3 * n)
    if mod_sym:
        for i in range(n):
            regmap["p%d" % i] = "%%%d" % (3 * n + i)
    for i in range(n):
        regmap["r%d" % i] = "%%%d" % i
        regmap["a%d" % i] = "%%%d" % (n + i)
        regmap["b%d" % i] = "%%%d" % (2 * n + i)
    body = pr.text(regmap)
    lines = []
    lines.append("__device__ __forceinline__ void %s(uint32_t* __restrict__ r, const uint32_t* a, const uint32_t* b) {" % fname)
    lines.append("  asm(\"{\\n\\t\"")
    lines.append("      \".reg .u32 e<%d>, o<%d>, mi, nm, hm, brw;\\n\\t\"" % (n, n))
    lines.append("      \".reg .pred %%pb;\\n\\t\"")
    for ln in body:
        lines.append("      \"%s\\n\\t\"" % ln.replace("%pb", "%%pb"))
    lines.append("      \"}\"")
    outs = ", ".join("\"=r\"(r[%d])" % i for i in range(n))
    ins = ", ".join("\"r\"(a[%d])" % i for i in range(n)) + ", " + ", ".join("\"r\"(b[%d])" % i for i in range(n))
    if mod_sym:
        ins += ", " + ", ".join("\"r\"(%s[%d])" % (mod_sym, i) for i in range(n))
    if m0_sym:
        ins += ", \"r\"(%s)" % m0_sym
    lines.append("      : %s" % outs)
    lines.append("      : %s);" % ins)
    lines.append("}")
    return "\n".join(lines)


def emit_fn_ops(fname, pr, n, operands):
    """General form: `operands` names the input arrays ("a", "b", "c", "d"; "a" alone for a square)."""
    regmap = {}
    for i in range(n):
        regmap["r%d" % i] = "%%%d" % i
        for k, nm in enumerate(operands):
            regmap["%s%d" % (nm, i)] = "%%%d" % ((k + 1) * n + i)
    if operands == ["a"]:
        for i in range(n):
            regmap["b%d" % i] = regmap["a%d" % i]
    body = pr.text(regmap)
    args = ", ".join("const uint32_t* %s" % nm for nm in operands)
    lines = ["__device__ __forceinline__ void %s(uint32_t* __restrict__ r, %s) {" % (fname, args)]
    lines.append("  asm(\"{\\n\\t\"")
    names = ["e<%d>" % n, "o<%d>" % n, "mi", "nm", "hm", "brw"] + list(dict.fromkeys(pr.temps))
    for k in range(0, len(names), 12):
        lines.append("      \".reg .u32 %s;\\n\\t\"" % ", ".join(names[k:k + 12]))
    lines.append("      \".reg .pred %%pb;\\n\\t\"")
    for ln in body:
        lines.append("      \"%s\\n\\t\"" % ln.replace("%pb", "%%pb"))
    lines.append("      \"}\"")
    outs = ", ".join("\"=r\"(r[%d])" % i for i in range(n))
    ins = ", ".join(", ".join("\"r\"(%s[%d])" % (nm, i) for i in range(n)) for nm in operands)
    lines.append("      : %s" % outs)
    lines.append("      : %s);" % ins)
    lines.append("}")
    return "\n".join(lines)


def check_sep(mod, n, trials=300):
    """wide-product + reduction forms (square, Karatsuba, lazy pairs) against big integers"""
    R = 1 << (32 * n)
    rinv = pow(R, -1, mod)
    rnd = random.Random(77 + n)
    edge = [0, 1, 2, mod - 1, mod - 2, (mod - 1) // 2, R % mod, (1 << (32 * n - 1)) % mod,
            ((1 << (16 * n)) - 1) % mod, ((((1 << (16 * n)) - 1) << (16 * n)) & (R - 1)) % mod]

    def run(pr, **vals):
        env = {}
        for nm, v in vals.items():
            for i, l in enumerate(limbs(v, n)):
                env["%s%d" % (nm, i)] = l
        out = pr.run(env)
        return sum(out["r%d" % i] << (32 * i) for i in range(n))

    pairs = [(x, y) for x in edge for y in edge] + [(rnd.randrange(mod), rnd.randrange(mod)) for _ in range(trials)]
    progs = {("mul", False): build_sep(mod, n, "mul"), ("mul", True): build_sep(mod, n, "mul", True),
             ("sqr", False): build_sep(mod, n, "sqr")}
    for x, y in pairs:
        assert run(progs[("mul", False)], a=x, b=y) == x * y * rinv % mod
        assert run(progs[("mul", True)], a=x, b=y) == x * y * rinv % mod
        assert run(progs[("sqr", False)], a=x, b=x) == x * x * rinv % mod
    if 3 * mod < R:  # a lazy pair needs the headroom (Fq: 381 of 384 bits; Fr has none)
        lazy = [build_mul(mod, n, pair2=True), build_sep(mod, n, "mul2"), build_sep(mod, n, "mul2", True)]
        quads = [(x, y, c, d) for x in edge[:6] for y in edge[:6] for c in edge[:6] for d in edge[:6]]
        quads += [tuple(rnd.randrange(mod) for _ in range(4)) for _ in range(trials)]
        for x, y, c, d in quads:
            for pr in lazy:
                assert run(pr, a=x, b=y, c=c, d=d) == (x * y + c * d) * rinv % mod
    print("%d-limb separated forms ok (%d pairs)" % (n, len(pairs)))


def main():
    check_sep(R_MOD, 8)
    check_sep(Q_MOD, 12)
    check_lazy(R_MOD, 8)
    check_lazy_fq(Q_MOD, 12)
    check("Fr", R_MOD, 8)
    check("Fr(mod in regs)", R_MOD, 8, mod_regs=True)
    check("Fr(m0 in a register)", R_MOD, 8, m0_reg=True)
    check("Fr(m0 in a register, low limbs by addition)", R_MOD, 8, m0_reg=True, special=True, trials=3000)
    check("Fq", Q_MOD, 12)
    if "--check-only" in sys.argv:
        return
    out = []
    out.append("// GENERATED by tools/gen_mont.py -- do not edit.  Inline-PTX Montgomery kernels for\n"
               "// BLS12-381 Fr (8 x u32) and Fq (12 x u32); carry chains validated by the generator's\n"
               "// CPU simulator against big-integer arithmetic.\n#pragma once\n#include <stdint.h>\n")
    def carr(x, n):
        return "{" + ", ".join("0x%08xu" % v for v in limbs(x, n)) + "}"
    for nm, mod, n in (("FR", R_MOD, 8), ("FQ", Q_MOD, 12)):
        R = (1 << (32 * n)) % mod
        out.append("#define TP_%s_MOD %s" % (nm, carr(mod, n)))
        out.append("#define TP_%s_ONE %s   // R mod p" % (nm, carr(R, n)))
        out.append("#define TP_%s_R2 %s   // R^2 mod p" % (nm, carr(R * R % mod, n)))
        out.append("#define TP_%s_MODM2 %s   // p - 2 (Fermat inversion exponent)" % (nm, carr(mod - 2, n)))
        if nm == "FQ":
            assert mod % 4 == 3
            out.append("#define TP_FQ_SQRT_EXP %s   // (q + 1) / 4 (square-root exponent, q = 3 mod 4)"
                       % carr((mod + 1) // 4, n))
    # Fr has -r^-1 mod 2^32 = 0xffffffff.  When ptxas sees that immediate it rewrites mi = -t0 and
    # then splits every reduction product mi * r_j into IMAD.X + IMAD.HI.U32.X (6.6 clk on the
    # FMA-heavy pipe instead of 4 for the fused IMAD.WIDE.U32.X) -- about half of all products of
    # the multiplication.  Feeding the constant through a __constant__ word keeps it opaque: 8 extra
    # 32-bit IMADs, all 128 products fused.  Fq's 0xfffcfffd does not trigger the rewrite.
    out.append("static __constant__ uint32_t TP_FR_M0 = 0xffffffffu;   // -r^-1 mod 2^32, deliberately not an immediate")
    for name, mod, n in (("fr", R_MOD, 8), ("fq", Q_MOD, 12)):
        if name == "fr":
            out.append(emit_fn("fr_mul_ptx", build_mul(mod, n, m0_reg=True, special=True), n, m0_sym="TP_FR_M0"))
            # lazy forms for the NTT butterflies (see build_add2): values in [0, 2r)
            out.append(emit_fn("fr_mul_lazy_ptx", build_mul(mod, n, reduce_final=False, m0_reg=True, special=True), n,
                               m0_sym="TP_FR_M0"))
            out.append(emit_fn("fr_add2_ptx", build_add2(mod, n), n))
            out.append(emit_fn("fr_sub2_ptx", build_sub(2 * mod, n), n))
            out.append(emit_fn_ops("fr_norm2_ptx", build_condsub(mod, n, (1,)), n, ["a"]))
        else:
            out.append(emit_fn("%s_mul_ptx" % name, build_mul(mod, n), n))
            # lazy pair a*b + c*d with one shared reduction (interleaved form: 432 products instead of 576)
            out.append(emit_fn_ops("fq_mul2_ptx", build_mul(mod, n, pair2=True), n, ["a", "b", "c", "d"]))
            # dedicated square: 78 + 144 products (wide product, then reduction)
            out.append(emit_fn_ops("fq_sqr_ptx", build_sep(mod, n, "sqr"), n, ["a"]))
            # separated forms kept for the multiplier microbenchmark (tools/ubench/fqmul_bench.cu)
            out.append(emit_fn_ops("fq_mul_sep_ptx", build_sep(mod, n, "mul"), n, ["a", "b"]))
            out.append(emit_fn_ops("fq_mul_kar_ptx", build_sep(mod, n, "mul", True), n, ["a", "b"]))
            out.append(emit_fn_ops("fq_mul2_kar_ptx", build_sep(mod, n, "mul2", True), n, ["a", "b", "c", "d"]))
            # lazy forms for the MSM's addition laws (see build_kq_minus): values in [0, 2q)
            out.append(emit_fn("fq_mul_lazy_ptx", build_mul(mod, n, reduce_final=False), n))
            out.append(emit_fn_ops("fq_mul2_lazy_ptx", build_mul(mod, n, reduce_final=False, pair2=True), n,
                                   ["a", "b", "c", "d"]))
            out.append(emit_fn_ops("fq_sqr_lazy_ptx", build_sep(mod, n, "sqr", reduce_final=False), n, ["a"]))
            out.append(emit_fn("fq_add2_ptx", build_add(2 * mod, n), n))
            out.append(emit_fn("fq_sub2_ptx", build_sub(2 * mod, n), n))
            out.append(emit_fn_ops("fq_neg1_ptx", build_kq_minus(mod, n, 1), n, ["a"]))
            out.append(emit_fn_ops("fq_neg2_ptx", build_kq_minus(mod, n, 2), n, ["a"]))
            out.append(emit_fn_ops("fq_norm2_ptx", build_condsub(mod, n, (1,)), n, ["a"]))
        out.append(emit_fn("%s_add_ptx" % name, build_add(mod, n), n))
        out.append(emit_fn("%s_sub_ptx" % name, build_sub(mod, n), n))
    dst = Path(__file__).resolve().parent.parent / "typlonk_b200" / "csrc" / "mont_gen.cuh"
    if "--out" in sys.argv:   # somewhere else (tests compare it with the committed header)
        dst = Path(sys.argv[sys.argv.index("--out") + 1])
    dst.parent.mkdir(parents=True, exist_ok=True)
    dst.write_text("\n\n".join(out) + "\n")
    print("wrote", dst)


if __name__ == "__main__":
    main()
