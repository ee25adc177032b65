"""CPU tests: the C restatement (oracle/c) against the Python-int oracle, bit for bit."""
import random

import numpy as np
import pytest

from oracle import binfmt as bf
from oracle import bn254 as bn
from oracle import cbind
from oracle import groth16 as g
from simple_zk_rollups_b200 import synth
from helpers import pack, pack_g1, pack_g2, unpack

R, Q = bn.R, bn.Q


def test_field_mul_kat():
    rng = random.Random(7)
    for field, p in ((0, Q), (1, R)):
        a = [0, 1, p - 1, (1 << 256) % p] + [rng.randrange(p) for _ in range(500)]
        b = [p - 1, p - 2, p - 1, 5] + [rng.randrange(p) for _ in range(500)]
        A, B = pack(a), pack(b)
        out = np.zeros_like(A)
        cbind.lib().oracle_field_mul(field, A.ctypes.data, B.ctypes.data, out.ctypes.data, len(a))
        rinv = pow(1 << 256, -1, p)
        assert unpack(out) == [x * y * rinv % p for x, y in zip(a, b)]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("nc,npub", [(5, 1), (80, 3), (400, 5)])
def test_c_prove_equals_python_prove(nc, npub, mode):
    r1, w = synth.generate(nc, npub, seed=nc + 1)
    pk, vk, _ = g.setup(r1.to_dicts(), (5, 4, 3, 2, 7))
    pkb, wb = bf.binarify_proving_key(pk), bf.binarify_witness(w)
    for r, s in ((0, 0), (R - 1, 12345)):
        want = g.proof_to_bytes(g.gen_proof(pk, w, r, s)[0])
        got, h = cbind.prove(pkb, wb, r, s, mode=mode, threads=3, want_h=True)
        assert got == want
        assert unpack(h) == g.calc_h_websnark(pk, w)


@pytest.mark.parametrize("group", [1, 2])
def test_c_msm_modes_agree_with_python(group):
    rng = random.Random(group)
    n = 300 if group == 1 else 120
    fb = bn.fixed_base(group)
    pts = fb.mul_many([rng.randrange(1, R) for _ in range(n)])
    pts[3] = None
    pts[9] = pts[8]
    sc = [0, 1, R - 1] + [rng.randrange(R) for _ in range(n - 3)]
    cur = bn.G1 if group == 1 else bn.G2
    want = cur.to_affine(g.msm_naive(cur, pts, sc))
    P = pack_g1(pts) if group == 1 else pack_g2(pts)
    for mode in (0, 1):
        out = unpack(np.frombuffer(cbind.msm(group, P, pack(sc), mode=mode, threads=4), dtype=np.uint8))
        got = (out[0], out[1]) if group == 1 else ((out[0], out[1]), (out[2], out[3]))
        assert got == want


def test_c_ntt_modes():
    rng = random.Random(3)
    for bits in (1, 4, 9, 13):
        x = [rng.randrange(R) for _ in range(1 << bits)]
        sh = g.root_of_unity(bits + 1)
        for mode in (0, 1):
            assert unpack(cbind.ntt(pack(x), bits, False, False, mode, 4)) == g.ntt(x)
            assert unpack(cbind.ntt(pack(x), bits, True, True, mode, 4)) == g.coset_intt(x, sh)


@pytest.mark.parametrize("bits", range(1, 11))
def test_c_h_from_evals(bits):
    """oracle_h_from_evals (websnark's 2m-point calcH, the host reference of the GPU H pipeline at every size) against
    the Python oracle's websnark and L/U methods, on full-range evaluations and on A_T = B_T = r - 1 (h = 0)."""
    rng = random.Random(50 + bits)
    m = 1 << bits
    at = [R - 1, 0, 1][:m] + [rng.randrange(R) for _ in range(m - 3)]
    bt = [rng.randrange(R) for _ in range(m - 1)] + [R - 1]
    pk = dict(domainSize=m, polsA=[{i: at[i] for i in range(m)}], polsB=[{i: bt[i] for i in range(m)}])
    want = g.calc_h_websnark(pk, [1])
    assert want == g.calc_h_lu(pk, [1])
    for mode in (0, 1):
        assert unpack(cbind.h_from_evals(pack(at), pack(bt), bits, mode=mode, threads=3)) == want
    assert not cbind.h_from_evals(pack([R - 1] * m), pack([R - 1] * m), bits).any()


@pytest.mark.parametrize("group", [1, 2])
def test_c_ap_points_equal_fixed_base(group):
    """oracle_ap_points (the host-side generator of the 2^20 arithmetic-progression MSM check) against per-point
    fixed-base multiplication on Python ints, including a step that walks through the point at infinity."""
    from helpers import unpack_g1, unpack_g2
    fb = bn.fixed_base(group)
    a0, d, n = 0x1234567, R - 3, 400
    base, step = fb.mul_many([a0, d])
    enc = (lambda pt: pack_g1([pt]).tobytes()) if group == 1 else (lambda pt: pack_g2([pt]).tobytes())
    got = cbind.ap_points(group, enc(base), enc(step), n)
    want = fb.mul_many([(a0 + i * d) % R for i in range(n)])
    assert (unpack_g1(got) if group == 1 else unpack_g2(got)) == want
    # (R - 2) G + i * G passes through infinity at i = 2 and through P == Q at i = 3
    base, step = fb.mul_many([R - 2, 1])
    got = cbind.ap_points(group, enc(base), enc(step), 6)
    want = fb.mul_many([(R - 2 + i) % R for i in range(6)])
    assert want[2] is None and (unpack_g1(got) if group == 1 else unpack_g2(got)) == want


def test_c_horner_and_exponent_sums():
    rng = random.Random(11)
    c = [0, R - 1] + [rng.randrange(R) for _ in range(300)]
    for x in (0, 1, R - 1, rng.randrange(R)):
        assert cbind.horner(pack(c), x) == sum(v * pow(x, j, R) for j, v in enumerate(c)) % R
    toxic = (0x1234567890ABCDEF1234567, 222222222222223, 3333333333333331, 44444444444447, 5555555555555557)
    for nc, npub in ((5, 1), (700, 5), (3000, 17)):
        r1, w = synth.generate(nc, npub, seed=nc)
        _, m = r1.domain()
        want = g.exponent_sums_flat(r1.with_input_rows(), r1.pool, npub, w, toxic, m)
        assert cbind.exponent_sums(r1.with_input_rows(), r1.pool, npub, synth.witness_bytes(w), toxic[0], m) == want
