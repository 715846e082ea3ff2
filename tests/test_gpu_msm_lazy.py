"""GPU: the MSM's lazy Fq arithmetic (tp_ctx_set_option "msm_fq_lazy", default 1: bucket state in [0, 2q), outputs
normalised before they leave the device) must give byte-identical commitments to the canonical laws ("msm_fq_lazy" = 0)
on one device and on sharded device groups (ranks on one device, as tests/test_gpu_multirank.py runs them): random
scalars (with and without the running-sum level of the reduction), all-equal scalars (one bucket per window holding
every point: the logarithmic boundary merge), buckets that receive P and -P, and repeated bases (doubling)."""
import random

import pytest

from oracle.pyoracle import curve, rng
from typlonk_b200 import field as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=[1, 2, 8])
def gctx(request, ctx):
    from typlonk_b200.ffi import Context
    if request.param == 1:
        yield ctx
        return
    g = Context.multi([0] * request.param)
    yield g
    g.close()


def both(c, srs, raw, **opts):
    """commitment with the lazy and with the canonical laws; the defaults are restored"""
    out = []
    try:
        for k, v in opts.items():
            c.set_option(k, v)
        for lazy in (1, 0):
            c.set_option("msm_fq_lazy", lazy)
            out.append(c.commit(srs, raw))
    finally:
        c.set_option("msm_fq_lazy", 1)
        for k in opts:
            c.set_option(k, 0)
    return out


def test_option_validation(ctx):
    from typlonk_b200.ffi import TyplonkError
    with pytest.raises(TyplonkError):
        ctx.set_option("msm_fq_lazy", 2)
    with pytest.raises(TyplonkError):
        ctx.set_option("msm_fq_lazy", -1)


@pytest.mark.parametrize("l1", [0, 1, 2])
def test_random_and_all_equal_scalars(gctx, l1):
    n = 70000
    tau = rng.fr_rand_stream(1, 1)[0]
    srs = gctx.srs_from_secret(F.fr_to_bytes(tau), n - 3)
    rnd = random.Random(11)
    cases = {
        "random": [rnd.randrange(F.R_MOD) for _ in range(n)],
        "all_equal": [0x1234567] * n,
        "r_minus_1": [F.R_MOD - 1] * n,
        "small": [rnd.randrange(1 << 12) for _ in range(n)],
    }
    for name, sc in cases.items():
        lazy, canon = both(gctx, srs, F.fr_vec_to_bytes(sc), msm_reduce_l1=l1)
        assert lazy == canon, (name, l1)
    srs.destroy()


def test_opposite_and_repeated_bases(gctx):
    g = curve.G1_GEN
    p2 = curve.g1_mul(g, 2)
    pts = [g, g, curve.g1_neg(g), p2, None, g, p2, p2] * 64
    srs = gctx.srs_upload(b"".join(F.g1_to_packed(p) for p in pts))
    n = len(pts)
    for sc in ([1] * n, [3] * n, list(range(1, n + 1)), [F.R_MOD - 1] * n, [2, 2, 2, 1] * (n // 4),
               [5 if i % 2 else F.R_MOD - 5 for i in range(n)]):
        raw = F.fr_vec_to_bytes(sc)
        lazy, canon = both(gctx, srs, raw)
        assert lazy == canon
        assert F.g1_from_abi(lazy) == curve.g1_msm(pts, F.fr_vec_from_bytes(raw))
    srs.destroy()
