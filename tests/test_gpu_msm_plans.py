"""GPU MSM at every window size and on both bucket-finishing paths, against host-only expectations.

The bases are multiples of the generator with known exponents, P_i = e_i G (e_i = 0: an infinity base), so every expected
sum is (sum k_i e_i mod r) G: Python ints and one scalar multiplication by the oracle, no GPU kernel.

Which code a shape runs (csrc/msm.cuh, msm_run): up to 20-bit windows the bucket partials are finished by the one-launch
gather (k_bucket_gather, whose whole-CTA path takes buckets with more than kHeavyRun = 48 level-1 partials); above, by the
recursive boundary levels (k_accum_xyzz while more than 4096 partials remain, big 4-per-thread branch from 2^16, then
k_accum_finish).  ZKR_MSM_LEVELS forces either, but is read once per process: the A/B arms run in child processes."""
import collections
import ctypes as C
import functools
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import bn254 as bn
from oracle import groth16 as g
from simple_zk_rollups_b200 import _lib
from helpers import affine_std, ap_points, check_ap_msm_full_size, pack, pack_g1, pack_g2, scalar_sets, unpack

pytestmark = pytest.mark.gpu
R = bn.R
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WINDOWS = list(range(2, 24))                 # every window size zkr_bases_load accepts
SWEEP_N = {1: 1000, 2: 450}                  # all_equal puts > 48 L entries into one bucket at every c (L = 8 or 16)


def n_windows(c):
    return (255 + c - 1) // c


def curve(group):
    return bn.G1 if group == 1 else bn.G2


def enc(group, pts):
    return pack_g1(pts) if group == 1 else pack_g2(pts)


@functools.lru_cache(maxsize=None)
def sweep_bases(group):
    """-> (exponents, points): random multiples of G with an infinity base at 3 and at n - 1, a duplicate (5 = 4) and a
    P / -P pair (7 = -4), as in test_gpu_msm.test_msm_small."""
    n = SWEEP_N[group]
    rng = random.Random(40 + group)
    e = [rng.randrange(1, R) for _ in range(n)]
    e[3] = e[n - 1] = 0
    e[5] = e[4]
    e[7] = R - e[4]
    return e, bn.fixed_base(group).mul_many(e)


def load(zctx, group, pts, c):
    L = _lib.lib()
    arr = enc(group, pts)
    h = C.c_void_p()
    _lib.check(L.zkr_bases_load(zctx, group, _lib.buf_ptr(arr), len(pts), c, C.byref(h)))
    cc, W = C.c_int(), C.c_int()
    _lib.check(L.zkr_bases_info(h, None, C.byref(cc), C.byref(W), None))
    assert c == 0 or (cc.value, W.value) == (c, n_windows(c))
    return h


def msm(zctx, group, h, scalars):
    out = np.zeros(64 if group == 1 else 128, dtype=np.uint8)
    sc = pack(scalars)
    _lib.check(_lib.lib().zkr_msm(zctx, h, _lib.buf_ptr(sc), len(scalars), 0, _lib.buf_ptr(out)))
    return affine_std(group, out)


def want(group, exps, scalars):
    return bn.fixed_base(group).mul_many([sum(k * e for k, e in zip(scalars, exps)) % R])[0]


# ------------------------------------------------------------------------------------------------ signed digits on the host
def signed_digits(k, c):
    """k_digits (csrc/msm.cuh) on Python ints: per window (|digit|, negative, carry in).  The digits must represent k
    and leave no carry out of the top window."""
    half, out, carry = 1 << (c - 1), [], 0
    for w in range(n_windows(c)):
        d, cin = ((k >> (c * w)) & ((1 << c) - 1)) + carry, carry
        carry = 0
        if d > half:
            d, carry = (1 << c) - d, 1
        out.append((d, carry == 1, cin))
    assert carry == 0 and sum((-d if neg else d) << (c * w) for w, (d, neg, _) in enumerate(out)) == k
    return out


def from_windows(c, low, top):
    """Scalar < r with the c-bit digits `low` in windows 0 .. W-2 and the top window's digit as close to `top` as r
    allows (low is cut to 253 bits first if it already reaches r: only at c = 2, whose top window holds no bit < 254)."""
    shift = c * (n_windows(c) - 1)
    k = sum(d << (c * w) for w, d in enumerate(low))
    if k >= R:
        k &= (1 << 253) - 1
    return k + (min(top, (R - 1 - k) >> shift) << shift)


def edge_scalars(c, n, rng):
    """One scalar per point, built window by window on the edges of k_digits: half = 2^(c-1) (the largest positive digit),
    half + 1 (negative, carries; repeated, the carry ripples through every window), 2^c - 1 (-1 with a carry; after a
    carry, a zero digit that still carries), with the top window's raw digit at 0, 1 or its largest value below r, plus
    r - 1, 2^253 and random scalars so that every bucket sees both signs."""
    W, half, full = n_windows(c), 1 << (c - 1), (1 << c) - 1
    edges = (0, 1, half - 1, half, half + 1, full - 1, full)
    fixed = [[half] * (W - 1), [half + 1] * (W - 1), [full] * (W - 1), [full, half] * W, [half + 1, half] * W]
    out = []
    for i in range(n):
        kind, top = i % 8, (0, 1, 1 << 30)[i // 8 % 3]
        if kind < len(fixed):
            out.append(from_windows(c, fixed[kind][:W - 1], top))
        elif kind == 5:
            out.append(from_windows(c, [rng.choice(edges) for _ in range(W - 1)], rng.choice((0, 1, half, 1 << 30))))
        else:
            out.append(rng.choice((R - 1, 1 << 253, rng.randrange(R))))
    return out


@pytest.mark.parametrize("c", WINDOWS)
@pytest.mark.parametrize("group", [1, 2])
def test_msm_every_window_size(zctx, group, c):
    """Forced window size c on points with infinities, duplicates and a P / -P pair; at c <= 20 the all_equal set goes
    through the gather's heavy-bucket path, at c >= 21 every set through the levels (k_accum_finish straight after
    level 1 at these sizes)."""
    exps, pts = sweep_bases(group)
    n = len(pts)
    compact = n - exps.count(0)
    # the heavy path is reached: one bucket holds more than kHeavyRun = 48 level-1 chunks of L entries (bases_build's L)
    total = n_windows(c) * compact
    L = 32 if total >= 1 << 22 else 16 if total >= 1 << 16 else 8
    sets = scalar_sets(random.Random(c * 10 + group), n)
    keys = collections.Counter(d - 1 for k, e in zip(sets["all_equal"], exps) if e for d, _, _ in signed_digits(k, c) if d)
    assert max(keys.values()) > 48 * L
    h = load(zctx, group, pts, c)
    for name, sc in sets.items():
        assert msm(zctx, group, h, sc) == want(group, exps, sc), name
    _lib.lib().zkr_bases_free(h)


@pytest.mark.parametrize("c", WINDOWS)
@pytest.mark.parametrize("group", [1, 2])
def test_msm_signed_digit_edges(zctx, group, c):
    """Scalars on every edge of the signed-digit recoding at window size c; scalars >= r are rejected with -3 and the
    range flag does not leak into the next MSM."""
    exps, pts = sweep_bases(group)
    n = len(pts)
    rng = random.Random(7000 + 100 * group + c)
    sc = edge_scalars(c, n, rng)
    assert all(0 <= k < R for k in sc)
    digits = [signed_digits(k, c) for k, e in zip(sc, exps) if e]
    W, half = n_windows(c), 1 << (c - 1)
    flat = [x for ds in digits for x in ds]
    assert any(d == half and not neg and cin == 0 for d, neg, cin in flat)          # largest positive digit, no carry
    assert any(d == half - 1 and neg for d, neg, _ in flat)                          # half + 1 -> negative, carries
    assert any(d == 0 and neg and cin for d, neg, cin in flat)                       # 2^c - 1 + carry -> zero, carries
    assert any(ds[-1][2] for ds in digits)                                           # carry into the short top window
    assert any(all(cin for _, _, cin in ds[1:W - 1]) for ds in digits)               # a carry through every window
    assert any(neg for d, neg, _ in flat if d) and any(not neg for d, neg, _ in flat if d)
    h = load(zctx, group, pts, c)
    assert msm(zctx, group, h, sc) == want(group, exps, sc)
    mixed = [rng.choice((k, R - 1, 1 << 253)) for k in sc]
    assert msm(zctx, group, h, mixed) == want(group, exps, mixed)
    assert exps[0]                                            # a scalar of an infinity base is never read
    for bad in (R, R + 1, 1 << 254, (1 << 256) - 1):
        with pytest.raises(_lib.ZkrError) as ei:
            msm(zctx, group, h, [bad] + sc[1:])
        assert ei.value.code == -3, hex(bad)
        assert msm(zctx, group, h, mixed) == want(group, exps, mixed), hex(bad)
    _lib.lib().zkr_bases_free(h)


@pytest.mark.parametrize("c", [2, 3, 21, 23])
@pytest.mark.parametrize("group", [1, 2])
def test_msm_tiny_against_naive(zctx, group, c):
    """A handful of points (mostly sentinel slots in the level-1 chunks) against the oracle's per-point double-and-add,
    which shares nothing with the exponent bookkeeping of the other tests."""
    rng = random.Random(300 + 10 * group + c)
    fb = bn.fixed_base(group)
    for n in (1, 2, 6):
        pts = fb.mul_many([rng.randrange(1, R) for _ in range(n)])
        if n == 6:
            pts[2], pts[3], pts[4] = None, pts[1], curve(group).neg(pts[0])
        h = load(zctx, group, pts, c)
        for sc in ([rng.randrange(R) for _ in range(n)], [R - 1] * n, [1 << 253] * n,
                   edge_scalars(c, n, rng)):
            assert msm(zctx, group, h, sc) == curve(group).to_affine(g.msm_naive(curve(group), pts, sc)), (n, sc)
        _lib.lib().zkr_bases_free(h)


@pytest.mark.parametrize("c", [2, 17, 23])
@pytest.mark.parametrize("group", [1, 2])
def test_window_table(zctx, group, c):
    """k_precompute: table[w n + i] == 2^(c w) P_i, byte for byte (affine, Montgomery), i over the compacted points."""
    exps, pts = sweep_bases(group)
    compact = [e for e in exps if e]
    n, W, AB = len(compact), n_windows(c), 64 if group == 1 else 128
    h = load(zctx, group, pts, c)
    fb = bn.fixed_base(group)
    for w in (0, 1, W - 1):
        for i in (0, 1, 3, 4, n // 2, n - 1):
            got = np.zeros(AB, dtype=np.uint8)
            _lib.check(_lib.lib().zkr_test_bases_peek(h, 0, AB * (w * n + i), _lib.buf_ptr(got), AB))
            assert got.tobytes() == enc(group, fb.mul_many([(compact[i] << (c * w)) % R])).tobytes(), (w, i)
    _lib.lib().zkr_bases_free(h)


# ------------------------------------------------------------------------------------------------ recursive levels at size
@pytest.mark.parametrize("group,log_n", [(1, 19), (2, 17)])
def test_msm_levels_full_size(zctx, group, log_n):
    """22-bit windows at 2^19 G1 / 2^17 G2 points: level 1 leaves more than 2^16 partials, so the levels run the big
    branch of level_log, then k_accum_xyzz, then k_accum_finish."""
    check_ap_msm_full_size(zctx, group, 1 << log_n, c=22)


def test_msm_levels_one_xyzz_level(zctx):
    """3000 G1 points at c = 22: 9216 level-1 partials, one k_accum_xyzz level, then k_accum_finish."""
    rng = random.Random(61)
    a0, d = rng.randrange(R), rng.randrange(R)
    n = 3000
    exps = [(a0 + i * d) % R for i in range(n)]
    h = load(zctx, 1, bn.fixed_base(1).mul_many(exps), 22)
    sets = scalar_sets(rng, n)
    sets["edges"] = edge_scalars(22, n, rng)
    for name, sc in sets.items():
        assert msm(zctx, 1, h, sc) == want(1, exps, sc), name
    _lib.lib().zkr_bases_free(h)


# ------------------------------------------------------------------------------------------------ ZKR_MSM_LEVELS arms
_CHILD = r"""
import ctypes as C, json, os, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from simple_zk_rollups_b200 import _lib
d, c = sys.argv[2], int(sys.argv[3])
L = _lib.lib()
ctx = C.c_void_p()
_lib.check(L.zkr_ctx_create(0, C.byref(ctx)))
res = {}
for job in json.load(open(os.path.join(d, "jobs.json"))):
    group, n = job["group"], job["n"]
    pts = np.fromfile(os.path.join(d, job["points"]), dtype=np.uint8)
    h, cc = C.c_void_p(), C.c_int()
    _lib.check(L.zkr_bases_load(ctx, group, _lib.buf_ptr(pts), n, c, C.byref(h)))
    _lib.check(L.zkr_bases_info(h, None, C.byref(cc), None, None))
    for name in job["scalars"]:
        sc = np.fromfile(os.path.join(d, name), dtype=np.uint8)
        out = np.zeros(64 if group == 1 else 128, dtype=np.uint8)
        _lib.check(L.zkr_msm(ctx, h, _lib.buf_ptr(sc), n, 0, _lib.buf_ptr(out)))
        res[name] = [cc.value, out.tobytes().hex()]
    L.zkr_bases_free(h)
L.zkr_ctx_destroy(ctx)
json.dump(res, open(os.path.join(d, "results.json"), "w"))
"""


def heavy_signed_scalars(c, n):
    """Thousands of heavy buckets of both signs: point i's digit magnitude j = 1 + (i / 2 mod n / 128) in every window,
    positive for even i, negative (with a carry, j - 1 above window 0) for odd i.  About 128 W entries per bucket."""
    W, m = n_windows(c), n // 128
    out = []
    for i in range(n):
        j = 1 + (i // 2) % m
        out.append(sum(j << (c * w) for w in range(W)) if i % 2 == 0 else
                   sum(((1 << c) - j) << (c * w) for w in range(W - 1)))
    return out


@pytest.mark.parametrize("levels,c", [(1, 17), (0, 22)], ids=["levels_at_c17", "gather_at_c22"])
def test_msm_levels_knob_arms(tmp_path, levels, c):
    """The arms of ZKR_MSM_LEVELS that no default plan takes: the recursive levels at 17-bit windows and the gather at
    22-bit windows (2^18 G1 points: 2048 heavy buckets for the whole-CTA path), each in a child process with its own
    context, since the knob is read once per process."""
    jobs, expect = [], {}
    for group, n in ((1, 1 << 18), (2, 1 << 15)):
        a0, d, pts = ap_points(group, n, random.Random(900 + group))
        pts.tofile(tmp_path / ("points_%d.bin" % group))
        rng = np.random.default_rng(group)
        uni = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        uni[:, 31] &= 0x1F                               # < 2^253 < r
        sets = {"uniform": [int.from_bytes(row.tobytes(), "little") for row in uni],
                "heavy_signed": heavy_signed_scalars(c, n),
                "all_equal": [0x1234567890ABCDEF1234567890ABCDEF] * n}
        for name, sc in sets.items():
            fname = "%s_%d.bin" % (name, group)
            pack(sc).tofile(tmp_path / fname)
            e = (a0 * sum(sc) + d * sum(i * k for i, k in enumerate(sc))) % R
            expect[fname] = (group, bn.fixed_base(group).mul_many([e])[0])
        jobs.append({"group": group, "n": n, "points": "points_%d.bin" % group,
                     "scalars": ["%s_%d.bin" % (name, group) for name in sets]})
    (tmp_path / "jobs.json").write_text(json.dumps(jobs))
    p = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path), str(c)], capture_output=True, text=True,
                       env=dict(os.environ, ZKR_MSM_LEVELS=str(levels)), timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    res = json.loads((tmp_path / "results.json").read_text())
    assert sorted(res) == sorted(expect)
    for fname, (group, pt) in expect.items():
        cc, out = res[fname]
        assert cc == c and affine_std(group, np.frombuffer(bytes.fromhex(out), dtype=np.uint8)) == pt, fname


# ------------------------------------------------------------------------------------------------ output forms, empty sets
def xyzz_to_affine(group, raw):
    """zkr_msm_dev's XYZZ bytes (X, Y, ZZ, ZZZ; Montgomery) -> oracle point: x = X / ZZ, y = Y / ZZZ."""
    rinv = pow(1 << 256, -1, bn.Q)
    v = [x * rinv % bn.Q for x in unpack(raw)]
    if group == 1:
        X, Y, ZZ, ZZZ = v
        if ZZ == 0:
            return None
        return X * bn.fq_inv(ZZ) % bn.Q, Y * bn.fq_inv(ZZZ) % bn.Q
    X, Y, ZZ, ZZZ = (v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7])
    if ZZ == (0, 0):
        return None
    return bn.f2_mul(X, bn.f2_inv(ZZ)), bn.f2_mul(Y, bn.f2_inv(ZZZ))


class DevBuf:
    def __init__(self, zctx, nbytes):
        self.zctx, self.p = zctx, C.c_void_p()
        _lib.check(_lib.lib().zkr_dev_malloc(zctx, nbytes, C.byref(self.p)))

    def free(self):
        _lib.check(_lib.lib().zkr_dev_free(self.zctx, self.p))


@pytest.mark.parametrize("c", [0, 22], ids=["default_plan", "levels_c22"])
@pytest.mark.parametrize("group", [1, 2])
def test_msm_output_forms(zctx, group, c):
    """zkr_msm_dev's XYZZ made affine on the host == zkr_msm's affine output == the expectation; device-resident scalars
    (scalars_on_device = 1) give the same result as host scalars, and an out-of-range one is rejected too."""
    L = _lib.lib()
    exps, pts = sweep_bases(group)
    n, XB, ob = len(pts), 128 if group == 1 else 256, 64 if group == 1 else 128
    h = load(zctx, group, pts, c)
    d_sc, d_out = DevBuf(zctx, 32 * n), DevBuf(zctx, XB)
    rng = random.Random(81 + group + c)
    for name, sc in scalar_sets(rng, n).items():
        exp = want(group, exps, sc)
        host = pack(sc)
        assert msm(zctx, group, h, sc) == exp, name
        _lib.check(L.zkr_dev_upload(zctx, d_sc.p, _lib.buf_ptr(host), host.size))
        out = np.zeros(ob, dtype=np.uint8)
        _lib.check(L.zkr_msm(zctx, h, d_sc.p, n, 1, _lib.buf_ptr(out)))
        assert affine_std(group, out) == exp, name
        raw = np.zeros(XB, dtype=np.uint8)
        _lib.check(L.zkr_msm_dev(zctx, h, d_sc.p, n, d_out.p))
        _lib.check(L.zkr_dev_download(zctx, _lib.buf_ptr(raw), d_out.p, XB))
        assert xyzz_to_affine(group, raw) == exp, name
    bad = pack([R] + [1] * (n - 1))
    _lib.check(L.zkr_dev_upload(zctx, d_sc.p, _lib.buf_ptr(bad), bad.size))
    with pytest.raises(_lib.ZkrError) as ei:
        _lib.check(L.zkr_msm(zctx, h, d_sc.p, n, 1, _lib.buf_ptr(out)))
    assert ei.value.code == -3
    d_sc.free()
    d_out.free()
    L.zkr_bases_free(h)


@pytest.mark.parametrize("group", [1, 2])
def test_msm_all_infinity_bases(zctx, group):
    """A base set of infinities only: zkr_msm writes zeros (infinity), zkr_msm_dev an XYZZ point with ZZ = ZZZ = 0."""
    L = _lib.lib()
    n, XB = 5, 128 if group == 1 else 256
    h = load(zctx, group, [None] * n, 0)
    npts = C.c_uint64()
    _lib.check(L.zkr_bases_info(h, C.byref(npts), None, None, None))
    assert npts.value == 0
    sc = pack([1, 2, R - 1, 1 << 253, 12345])
    out = np.full(64 if group == 1 else 128, 0xAB, dtype=np.uint8)
    _lib.check(L.zkr_msm(zctx, h, _lib.buf_ptr(sc), n, 0, _lib.buf_ptr(out)))
    assert not out.any()
    d_sc, d_out = DevBuf(zctx, 32 * n), DevBuf(zctx, XB)
    _lib.check(L.zkr_dev_upload(zctx, d_sc.p, _lib.buf_ptr(sc), sc.size))
    raw = np.full(XB, 0xAB, dtype=np.uint8)
    _lib.check(L.zkr_dev_upload(zctx, d_out.p, _lib.buf_ptr(raw), XB))
    _lib.check(L.zkr_msm_dev(zctx, h, d_sc.p, n, d_out.p))
    _lib.check(L.zkr_dev_download(zctx, _lib.buf_ptr(raw), d_out.p, XB))
    assert not raw[XB // 2:].any()                            # ZZ and ZZZ: the identity
    d_sc.free()
    d_out.free()
    L.zkr_bases_free(h)
