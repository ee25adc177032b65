"""GPU parity: bucketed MSM (G1 and G2) vs the oracle's per-point double-and-add, bit-exact."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import bn254 as bn
from oracle import groth16 as g
from simple_zk_rollups_b200 import _lib
from helpers import check_ap_msm_full_size, pack, pack_g1, pack_g2, scalar_sets, unpack

pytestmark = pytest.mark.gpu
R = bn.R


def _with_lazy(value):
    import os
    old = os.environ.get("ZKR_LAZY")
    os.environ["ZKR_LAZY"] = str(value)
    yield value
    if old is None:
        del os.environ["ZKR_LAZY"]
    else:
        os.environ["ZKR_LAZY"] = old


@pytest.fixture(params=[0, 7], ids=["madd", "madd_lazy_sqr"])
def lazy(request):
    """The round-1 form and the default form of the bucket accumulation's mixed addition (ZKR_LAZY is read on every MSM
    call; csrc/msm.cuh): 0 = plain, 7 = sums of products reduced once + dedicated squaring."""
    yield from _with_lazy(request.param)


@pytest.fixture
def lazy_intermediate():
    """3 = sums of products reduced once, generic squaring (the A/B's middle arm stays selectable, so it stays tested)"""
    yield from _with_lazy(3)


def load_bases(zctx, group, pts, c=0):
    L = _lib.lib()
    arr = pack_g1(pts) if group == 1 else pack_g2(pts)
    h = C.c_void_p()
    _lib.check(L.zkr_bases_load(zctx, group, _lib.buf_ptr(arr), len(pts), c, C.byref(h)))
    return h


def msm(zctx, group, h, scalars):
    L = _lib.lib()
    sc = pack(scalars)
    out = np.zeros(64 if group == 1 else 128, dtype=np.uint8)
    _lib.check(L.zkr_msm(zctx, h, _lib.buf_ptr(sc), len(scalars), 0, _lib.buf_ptr(out)))
    v = unpack(out)
    if not any(v):
        return None
    return (v[0], v[1]) if group == 1 else ((v[0], v[1]), (v[2], v[3]))


def want(group, pts, scalars):
    cur = bn.G1 if group == 1 else bn.G2
    return cur.to_affine(g.msm_naive(cur, pts, scalars))


@pytest.mark.parametrize("group,n,c", [(1, 1, 0), (1, 2, 4), (1, 37, 0), (1, 300, 5), (1, 300, 13), (1, 1500, 0),
                                       (2, 1, 0), (2, 41, 4), (2, 200, 0), (2, 200, 11)])
def test_msm_small(zctx, group, n, c, lazy):
    L = _lib.lib()
    rng = random.Random(1000 * group + n + c)
    fb = bn.fixed_base(group)
    pts = fb.mul_many([rng.randrange(1, R) for _ in range(n)])
    if n > 5:
        pts[3] = None                         # infinity bases are skipped (B1/B2 of absent signals)
        pts[n - 1] = None
        pts[5] = pts[4]                       # duplicate bases -> P == Q inside a bucket
        cur = bn.G1 if group == 1 else bn.G2
        pts[7 % n] = cur.neg(pts[4])          # and P == -Q
    h = load_bases(zctx, group, pts, c)
    npts, cc, W, nbytes = C.c_uint64(), C.c_int(), C.c_int(), C.c_uint64()
    _lib.check(L.zkr_bases_info(h, C.byref(npts), C.byref(cc), C.byref(W), C.byref(nbytes)))
    assert npts.value == sum(p is not None for p in pts) and (c == 0 or cc.value == c)
    for name, sc in scalar_sets(rng, n).items():
        assert msm(zctx, group, h, sc) == want(group, pts, sc), "%s (c=%d W=%d)" % (name, cc.value, W.value)
    # out-of-range scalar is rejected, not reduced
    bad = [R] + [1] * (n - 1)
    if pts[0] is not None:
        with pytest.raises(_lib.ZkrError) as ei:
            msm(zctx, group, h, bad)
        assert ei.value.code == -3
    L.zkr_bases_free(h)


@pytest.mark.parametrize("group,n", [(1, 3000), (2, 800)])
def test_msm_intermediate_accumulation_form(zctx, group, n, lazy_intermediate):
    rng = random.Random(5 + group)
    a0, d = rng.randrange(R), rng.randrange(R)
    fb = bn.fixed_base(group)
    pts = fb.mul_many([(a0 + i * d) % R for i in range(n)])
    h = load_bases(zctx, group, pts)
    for name in ("uniform", "rollup_like", "all_equal"):
        sc = scalar_sets(rng, n)[name]
        e = sum(k * (a0 + i * d) for i, k in enumerate(sc)) % R
        assert msm(zctx, group, h, sc) == fb.mul_many([e])[0], name
    _lib.lib().zkr_bases_free(h)


@pytest.mark.parametrize("group,n", [(1, 30000), (2, 6000)])
def test_msm_arithmetic_progression(zctx, group, n, lazy):
    """P_i = (a0 + i d) G  =>  sum k_i P_i = (sum k_i (a0 + i d) mod r) G   (SURVEY 8(d) config 3 check)."""
    L = _lib.lib()
    rng = random.Random(77 + group)
    a0, d = rng.randrange(R), rng.randrange(R)
    fb = bn.fixed_base(group)
    pts = fb.mul_many([(a0 + i * d) % R for i in range(n)])
    h = load_bases(zctx, group, pts)
    for name, sc in scalar_sets(rng, n).items():
        if name in ("half_window",):
            continue
        e = sum(k * (a0 + i * d) for i, k in enumerate(sc)) % R
        exp = fb.mul_many([e])[0]
        assert msm(zctx, group, h, sc) == exp, name
    L.zkr_bases_free(h)


@pytest.mark.parametrize("group,log_n", [(1, 20), (2, 17)])
def test_msm_arithmetic_progression_full_size(zctx, group, log_n):
    """SURVEY 8(d) config 3 at 2^20 (G1) / 2^17 (G2) with a HOST-ONLY expectation: the points P_i = (a0 + i d) G come
    from the oracle's C restatement (a chain of additions, no GPU), the expected sum is (sum k_i (a0 + i d) mod r) G
    on Python ints.  Scalar sets: uniform, rollup-like (3 % in {0, 1}) and every adversarial set of config 3 (iii)."""
    check_ap_msm_full_size(zctx, group, 1 << log_n)
