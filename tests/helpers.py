"""Byte-level packing helpers and host-only MSM expectations shared by the GPU parity tests."""
import ctypes as C
import random

import numpy as np

from oracle import bn254 as bn

MONT = 1 << 256
R = bn.R


def pack(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint8).copy()


def unpack(arr):
    b = arr.tobytes()
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def pack_g1(pts):
    return pack([c * MONT % bn.Q for p in pts for c in ((0, 0) if p is None else p)])


def pack_g2(pts):
    flat = []
    for p in pts:
        flat += [0, 0, 0, 0] if p is None else [p[0][0], p[0][1], p[1][0], p[1][1]]
    return pack([c * MONT % bn.Q for c in flat])


def unpack_g1(arr):
    rinv = pow(MONT, -1, bn.Q)
    v = [x * rinv % bn.Q for x in unpack(arr)]
    return [None if (v[i] == 0 and v[i + 1] == 0) else (v[i], v[i + 1]) for i in range(0, len(v), 2)]


def unpack_g2(arr):
    rinv = pow(MONT, -1, bn.Q)
    v = [x * rinv % bn.Q for x in unpack(arr)]
    return [None if not any(v[i:i + 4]) else ((v[i], v[i + 1]), (v[i + 2], v[i + 3])) for i in range(0, len(v), 4)]


def affine_std(group, out):
    """zkr_msm's output bytes (affine, standard form; all zeros = infinity) -> oracle point"""
    v = unpack(out)
    if not any(v):
        return None
    return (v[0], v[1]) if group == 1 else ((v[0], v[1]), (v[2], v[3]))


def scalar_sets(rng, n):
    half = n // 2
    return {
        "uniform": [rng.randrange(R) for _ in range(n)],
        "rollup_like": [rng.choice((0, 1)) if rng.random() < 0.3 else rng.randrange(R) for _ in range(n)],
        "all_zero": [0] * n,
        "all_one": [1] * n,
        "all_rm1": [R - 1] * n,
        "all_equal": [0x1234567890ABCDEF1234567890ABCDEF % R] * n,
        "alternating": [(7 if i % 2 == 0 else R - 7) for i in range(n)],
        "small": [rng.randrange(1 << 16) for _ in range(n)],
        "half_window": [(1 << (rng.randrange(1, 250))) for _ in range(half)] + [rng.randrange(R) for _ in range(n - half)],
    }


def ap_points(group, n, rng):
    """P_i = (a0 + i d) G, i < n, with random a0, d: -> (a0, d, n x 64 / 128 B affine Fq-M points).  The points come
    from the oracle's C restatement (a chain of additions, no GPU); three of them are checked against points computed
    independently."""
    from oracle import cbind
    a0, d = rng.randrange(R), rng.randrange(R)
    fb = bn.fixed_base(group)
    enc = (lambda pt: pack_g1([pt]).tobytes()) if group == 1 else (lambda pt: pack_g2([pt]).tobytes())
    base, step = fb.mul_many([a0, d])
    pts = cbind.ap_points(group, enc(base), enc(step), n)
    width = 64 if group == 1 else 128
    for i in (0, 1, n - 1):
        assert pts[width * i:width * (i + 1)].tobytes() == enc(fb.mul_many([(a0 + i * d) % R])[0])
    return a0, d, pts


def check_ap_msm_full_size(zctx, group, n, c=0):
    """SURVEY 8(d) config 3 with a HOST-ONLY expectation: on P_i = (a0 + i d) G (ap_points) the expected sum is
    (sum k_i (a0 + i d) mod r) G on Python ints.  Scalar sets: uniform, rollup-like (3 % in {0, 1}) and every
    adversarial set of config 3 (iii).  c > 0 forces the window size."""
    from simple_zk_rollups_b200 import _lib
    L = _lib.lib()
    a0, d, pts = ap_points(group, n, random.Random(500 + group))
    fb = bn.fixed_base(group)
    h = C.c_void_p()
    _lib.check(L.zkr_bases_load(zctx, group, _lib.buf_ptr(pts), n, c, C.byref(h)))
    if c:
        cc = C.c_int()
        _lib.check(L.zkr_bases_info(h, None, C.byref(cc), None, None))
        assert cc.value == c
    s1 = n * (n - 1) // 2                       # sum i
    k_eq = 0x1234567890ABCDEF1234567890ABCDEF % R
    uni = np.random.default_rng(9).integers(0, 256, size=(n, 32), dtype=np.uint8)
    uni[:, 31] &= 0x1F                          # < 2^253 < r
    roll = uni.copy()
    sel = np.random.default_rng(10).random(n) < 0.03
    roll[sel] = 0
    roll[sel, 0] = np.random.default_rng(11).integers(0, 2, size=int(sel.sum()), dtype=np.uint8)

    def dot(arr):                               # sum k_i (a0 + i d) on Python ints
        ks = [int.from_bytes(arr[i].tobytes(), "little") for i in range(n)]
        return (a0 * sum(ks) + d * sum(i * k for i, k in enumerate(ks))) % R

    const = lambda k: np.tile(np.frombuffer(int(k).to_bytes(32, "little"), dtype=np.uint8), (n, 1))
    alt = const(7)
    alt[1::2] = np.frombuffer(int(R - 7).to_bytes(32, "little"), dtype=np.uint8)
    cases = {
        "uniform": (uni, None), "rollup_like": (roll, None),
        "all_zero": (const(0), 0), "all_one": (const(1), (a0 * n + d * s1) % R),
        "all_rm1": (const(R - 1), (R - 1) * (a0 * n + d * s1) % R),
        "all_equal": (const(k_eq), k_eq * (a0 * n + d * s1) % R),
        "alternating": (alt, None),
    }
    width = 64 if group == 1 else 128
    for name, (arr, e) in cases.items():
        if e is None:
            e = dot(arr)
        out = np.zeros(width, dtype=np.uint8)
        sc = np.ascontiguousarray(arr).reshape(-1)
        _lib.check(L.zkr_msm(zctx, h, _lib.buf_ptr(sc), n, 0, _lib.buf_ptr(out)))
        assert affine_std(group, out) == fb.mul_many([e])[0], name
    L.zkr_bases_free(h)
