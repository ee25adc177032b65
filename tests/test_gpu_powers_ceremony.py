"""Phase-1 powers of tau (csrc/powers.cu, zkr.h "phase 1"): contributions, their records and the verifiers.

A contribution is deterministic in its secrets, so it is checked byte for byte: contributing (tau', alpha', beta') to
the powers of (tau, alpha, beta) must give the powers of (tau tau', alpha alpha', beta beta').  Synthetic powers come
from scalars computed with Python ints and turned into points by zkr_synth_points.  The records are re-derived with
hashlib and checked on the oracle's integer curve arithmetic."""
import hashlib
import random

import numpy as np
import pytest

from oracle import bn254 as bn
from simple_zk_rollups_b200 import _lib, keygen, prover, synth

R, Q = bn.R, bn.Q
RINV_Q = pow(1 << 256, -1, Q)
NAMES = ("tau", "alpha", "beta")

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gp():
    p = prover.Groth16Prover(0)
    yield p
    p.close()


def _points(ctx, group, scalars):
    sc = np.frombuffer(b"".join(int(s % R).to_bytes(32, "little") for s in scalars), dtype=np.uint8)
    out = np.empty(len(scalars) * (64 if group == 1 else 128), dtype=np.uint8)
    _lib.check(_lib.lib().zkr_synth_points(ctx, group, _lib.buf_ptr(sc), len(scalars), _lib.buf_ptr(out)))
    return out.tobytes()


def _pows(x, n, c=1):
    out, acc = [], c % R
    for _ in range(n):
        out.append(acc)
        acc = acc * x % R
    return out


def powers(ctx, tau, alpha, beta, n_g1, n_g2, n_a=None, n_b=None):
    """Phase-1 points of (tau, alpha, beta) with the given counts (alpha / beta default to n_g2)."""
    n_a = n_g2 if n_a is None else n_a
    n_b = n_g2 if n_b is None else n_b
    return {"tau_g1": _points(ctx, 1, _pows(tau, n_g1)), "tau_g2": _points(ctx, 2, _pows(tau, n_g2)),
            "alpha_tau_g1": _points(ctx, 1, _pows(tau, n_a, alpha)), "beta_tau_g1": _points(ctx, 1, _pows(tau, n_b, beta)),
            "beta_g2": _points(ctx, 2, [beta])}


def counts(p):
    return (len(p["tau_g1"]) // 64, len(p["tau_g2"]) // 128, len(p["alpha_tau_g1"]) // 64, len(p["beta_tau_g1"]) // 64)


def assert_same_powers(got, want):
    for name, size in (("tau_g1", 64), ("tau_g2", 128), ("alpha_tau_g1", 64), ("beta_tau_g1", 64), ("beta_g2", 128)):
        a, b = bytes(got[name]), bytes(want[name])
        assert len(a) == len(b), name
        if a != b:
            first = next(i for i in range(len(a)) if a[i] != b[i])
            pytest.fail("%s differs first at point %d" % (name, first // size))


def secrets(seed):
    rng = random.Random(seed)
    return [rng.randrange(1, R) for _ in range(3)]


def check_contribution(ctx, shape, old_secrets, new_secrets):
    """powers_contribute(powers(old), new) == powers(old * new), for the counts `shape`."""
    old = powers(ctx, *old_secrets, *shape)
    got, rec = keygen.powers_contribute(ctx, old, *new_secrets)
    assert len(rec) == _lib.POWERS_RECORD_BYTES
    assert_same_powers(got, powers(ctx, *[a * b % R for a, b in zip(old_secrets, new_secrets)], *shape))
    return old, got, rec


# ------------------------------------------------------------------------------------------------ byte identity
@pytest.mark.parametrize("log_m", range(1, 13))
def test_contribution_is_byte_identical(gp, log_m):
    m = 1 << log_m
    check_contribution(gp.ctx, (2 * m, m), secrets(log_m), secrets(100 + log_m))


@pytest.mark.parametrize("shape", [(2, 2, 1, 1), (3, 5, 1, 1), (199, 100, 1, 1), (205, 103, 1, 1), (37, 2, 7, 1)])
def test_unequal_counts_are_byte_identical(gp, shape):
    """n_tau_g1 = 2, 3, 2m - 1, 2m + 5 for m = 100; alpha and beta of one point; nothing assumes 2^K."""
    check_contribution(gp.ctx, shape, secrets(shape[0]), secrets(shape[1] + 7))


TOP = (0x2F << 248) | ((1 << 248) - 1)      # nibble 62 is 0xf: the signed-window recoding carries into the top window


@pytest.mark.parametrize("new", [(1, 5, 7), (R - 1, 3, 4), (123456789, 1, 1), (TOP, TOP, TOP), (1, 1, 1), (R - 1, R - 1, R - 1)],
                         ids=["tau1", "tau_r-1", "alpha_beta_1", "top_window_carry", "all1", "all_r-1"])
def test_edge_secrets(gp, new):
    assert TOP < R
    old, got, _ = check_contribution(gp.ctx, (70, 33), secrets(5), new)
    if new[0] == R - 1:          # tau' = -1: powers alternate between P and -P
        t0, t1 = np.frombuffer(old["tau_g1"], dtype=np.uint8).reshape(-1, 64), np.frombuffer(got["tau_g1"], dtype=np.uint8).reshape(-1, 64)
        assert (t1[0::2] == t0[0::2]).all()
        y0 = [int.from_bytes(bytes(r[32:]), "little") for r in t0[1::2]]
        y1 = [int.from_bytes(bytes(r[32:]), "little") for r in t1[1::2]]
        assert all((a + b) % Q == 0 for a, b in zip(y0, y1))
    if new == (1, 1, 1):
        assert_same_powers(got, old)


@pytest.fixture(scope="module")
def big(gp):
    """The 2^20 rollup shape's ceremony (2^21 G1 powers, 2^20 of the others) and one contribution to it."""
    m = 1 << 20
    old_s, new_s = secrets(20), secrets(21)
    old, got, rec = check_contribution(gp.ctx, (2 * m, m), old_s, new_s)
    return dict(old=old, new=got, rec=rec)


def test_rollup_shapes_are_byte_identical(gp, big):
    m = 1 << 17                                          # tx.circom's domain; the 2^20 shape is the `big` fixture
    check_contribution(gp.ctx, (2 * m, m), secrets(17), secrets(18))
    assert counts(big["new"]) == (1 << 21, 1 << 20, 1 << 20, 1 << 20)


# ------------------------------------------------------------------------------------------------ chain
def test_chain_to_a_proof(gp):
    """powers_new -> two verified contributions -> setup_from_powers -> phase-2 contribution: the key of
    synth_setup(tau1 tau2, alpha1 alpha2, beta1 beta2, 1, delta), and its proofs."""
    r1, w = synth.generate(300, 4, seed=5)
    bits, m = r1.domain()
    p0 = keygen.powers_new(gp.ctx, m)
    assert keygen.powers_verify(gp.ctx, p0) == (True, "")
    s1, s2 = secrets(31), secrets(32)
    p1, rec1 = keygen.powers_contribute(gp.ctx, p0, *s1)
    assert keygen.powers_verify_contribution(gp.ctx, p0, p1, rec1) == (True, "")
    p2, rec2 = keygen.powers_contribute(gp.ctx, p1, *s2)
    assert keygen.powers_verify_contribution(gp.ctx, p1, p2, rec2) == (True, "")
    tau, alpha, beta = (a * b % R for a, b in zip(s1, s2))
    pk, vk = keygen.setup_from_powers(gp.ctx, r1, p2)
    d = 8675309
    pk1, vk1, rec = keygen.contribute(gp.ctx, pk, vk, d)
    assert keygen.verify_contribution(gp.ctx, pk, vk, pk1, vk1, rec)
    ref_pk, ref_vk = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, d))
    assert bytes(pk1) == bytes(ref_pk) and bytes(vk1["bin"]) == bytes(ref_vk["bin"])
    pa, _ = gp.prove(gp.load_key(pk1), synth.witness_bytes(w), 21, 22)
    pb, _ = gp.prove(gp.load_key(ref_pk), synth.witness_bytes(w), 21, 22)
    assert pa == pb
    assert gp.verify(gp.load_vkey(vk1["bin"]), pa, w[1:5])


# ------------------------------------------------------------------------------------------------ record
def _g1(b):
    x = int.from_bytes(b[:32], "little") * RINV_Q % Q
    y = int.from_bytes(b[32:64], "little") * RINV_Q % Q
    return None if x == 0 else (x, y)


def _bases(p):
    return [bytes(p["tau_g1"][64:128]), bytes(p["alpha_tau_g1"][:64]), bytes(p["beta_tau_g1"][:64])]


def test_record_pinned_from_outside(gp):
    """c = SHA-256("zkr-phase1-" name | P_old | P_new | R) mod r, P_new = s' P_old and z P_old = R + c P_new on oracle
    integers; with a known s', R = (z - c s') P_old."""
    new_s = (424242424242, 98765, 55555)
    old, new, rec = check_contribution(gp.ctx, (16, 8), secrets(77), new_s)
    for j, (po, pn) in enumerate(zip(_bases(old), _bases(new))):
        Rb, z = rec[96 * j:96 * j + 64], int.from_bytes(rec[96 * j + 64:96 * j + 96], "little")
        assert z < R
        c = int.from_bytes(hashlib.sha256(b"zkr-phase1-" + NAMES[j].encode() + po + pn + Rb).digest(), "little") % R
        P_old, P_new, P_R = _g1(po), _g1(pn), _g1(Rb)
        assert P_new == bn.G1.mul(P_old, new_s[j])
        assert bn.G1.mul(P_old, z) == bn.G1.add(P_R, bn.G1.mul(P_new, c))
        assert P_R == bn.G1.mul(P_old, (z - c * new_s[j]) % R)


# ------------------------------------------------------------------------------------------------ powers_verify
def _replace(p, name, idx, data):
    size = 128 if name in ("tau_g2", "beta_g2") else 64
    b = bytearray(p[name])
    b[idx * size:idx * size + len(data)] = data
    q = dict(p)
    q[name] = bytes(b)
    return q


def _mont(v):
    return (v * (1 << 256) % Q).to_bytes(32, "little")


def _f2_pow(a, e):
    r = bn.F2_ONE
    while e:
        if e & 1:
            r = bn.f2_mul(r, a)
        a = bn.f2_sqr(a)
        e >>= 1
    return r


def _f2_sqrt(a):
    """square root in Fq2 for q = 3 mod 4 (None if a is a non-residue)"""
    a1 = _f2_pow(a, (Q - 3) // 4)
    alpha = bn.f2_mul(bn.f2_sqr(a1), a)
    if bn.f2_mul(bn.f2_conj(alpha), alpha) == ((Q - 1) % Q, 0):
        return None
    x0 = bn.f2_mul(a1, a)
    if alpha == ((Q - 1) % Q, 0):
        x = bn.f2_mul((0, 1), x0)
    else:
        x = bn.f2_mul(_f2_pow(bn.f2_add(bn.F2_ONE, alpha), (Q - 1) // 2), x0)
    return x if bn.f2_sqr(x) == a else None


def _twist_point_outside_subgroup():
    """on the twist but outside the order-r subgroup (the twist has a large cofactor): first x = 1, 2, .. with a root"""
    for x in range(1, 60):
        y = _f2_sqrt(bn.f2_add(bn.f2_mul(bn.f2_sqr((x, 0)), (x, 0)), bn.B2))
        if y is not None:
            pt = ((x, 0), y)
            assert bn.G2.is_on_curve(pt) and not bn.g2_in_subgroup(pt)
            return _mont(x) + _mont(0) + _mont(y[0]) + _mont(y[1])
    raise AssertionError("no point found")


def _rejected(ctx, p, reason):
    ok, why = keygen.powers_verify(ctx, p)
    assert not ok
    assert reason in why, why


def test_verify_accepts(gp, big):
    assert keygen.powers_verify(gp.ctx, keygen.powers_new(gp.ctx, 16)) == (True, "")
    assert keygen.powers_verify(gp.ctx, keygen.powers_new(gp.ctx, 4, n_tau_g1=5)) == (True, "")
    for shape in ((128, 64), (2, 2, 1, 1), (41, 9, 3, 17)):
        assert keygen.powers_verify(gp.ctx, powers(gp.ctx, *secrets(len(shape)), *shape)) == (True, "")
    assert keygen.powers_verify(gp.ctx, big["new"]) == (True, "")


def test_verify_rejects(gp):
    m = 64
    tau, alpha, beta = secrets(3)
    p = powers(gp.ctx, tau, alpha, beta, 2 * m, m)
    assert keygen.powers_verify(gp.ctx, p) == (True, "")
    other = _points(gp.ctx, 1, [987654321])
    for idx in (1, m, 2 * m - 1):              # another valid point at index 1, in the middle, last
        _rejected(gp.ctx, _replace(p, "tau_g1", idx, other), "G1 same-ratio check failed")
    t = bytearray(p["tau_g1"])
    t[64 * 5:64 * 6], t[64 * 6:64 * 7] = t[64 * 6:64 * 7], t[64 * 5:64 * 6]
    _rejected(gp.ctx, dict(p, tau_g1=bytes(t)), "G1 same-ratio check failed")
    _rejected(gp.ctx, dict(p, alpha_tau_g1=_points(gp.ctx, 1, _pows(tau + 1, m, alpha))), "G1 same-ratio check failed")
    _rejected(gp.ctx, _replace(p, "beta_tau_g1", m - 1, other), "G1 same-ratio check failed")
    _rejected(gp.ctx, _replace(p, "tau_g2", m // 2, _points(gp.ctx, 2, [5])), "G2 same-ratio check failed")
    _rejected(gp.ctx, dict(p, beta_g2=_points(gp.ctx, 2, [beta + 1])), "beta_tau_g1[0] and beta_g2 have different beta")
    _rejected(gp.ctx, _replace(p, "tau_g1", 0, _points(gp.ctx, 1, [2])), "tau_g1[0] is not the G1 generator")
    _rejected(gp.ctx, _replace(p, "tau_g2", 0, _points(gp.ctx, 2, [2])), "tau_g2[0] is not the G2 generator")
    bad2 = _twist_point_outside_subgroup()
    _rejected(gp.ctx, _replace(p, "tau_g2", 5, bad2), "tau_g2[5] is not in the order-r subgroup")
    _rejected(gp.ctx, dict(p, beta_g2=bad2), "beta_g2[0] is not in the order-r subgroup")
    _rejected(gp.ctx, _replace(p, "tau_g1", 9, p["tau_g1"][9 * 64:9 * 64 + 32] + _mont(5)), "tau_g1[9] is not on the curve")
    _rejected(gp.ctx, _replace(p, "alpha_tau_g1", 3, Q.to_bytes(32, "little")), "alpha_tau_g1[3] has a coordinate >= q")
    _rejected(gp.ctx, _replace(p, "tau_g2", 7, b"\0" * 64), "tau_g2[7] is the point at infinity")
    # the first failing point is reported
    q = _replace(_replace(p, "beta_tau_g1", 40, b"\0" * 32), "beta_tau_g1", 30, b"\0" * 32)
    _rejected(gp.ctx, q, "beta_tau_g1[30] is the point at infinity")


def test_verify_rejects_one_tamper_among_2p21(gp, big):
    p = big["new"]
    n = counts(p)[0]
    _rejected(gp.ctx, _replace(p, "tau_g1", n // 2 + 12345, _points(gp.ctx, 1, [31337])), "G1 same-ratio check failed")


def test_verify_in_slices(gp):
    """n_tau_g1 = 2^22 + 5: the MSM bases are loaded in two slices; a tamper in the last slice is found."""
    tau, alpha, beta = secrets(22)
    n = (1 << 22) + 5
    p = powers(gp.ctx, tau, alpha, beta, n, 4)
    assert keygen.powers_verify(gp.ctx, p) == (True, "")
    _rejected(gp.ctx, _replace(p, "tau_g1", n - 3, _points(gp.ctx, 1, [7])), "G1 same-ratio check failed")
    # the pair that straddles the slice boundary is checked as well
    _rejected(gp.ctx, _replace(p, "tau_g1", 1 << 22, _points(gp.ctx, 1, [7])), "G1 same-ratio check failed")


# ------------------------------------------------------------------------------------------------ verify_contribution
@pytest.fixture(scope="module")
def link(gp):
    shape = (40, 20)
    old_s, new_s = secrets(50), secrets(51)
    old, new, rec = check_contribution(gp.ctx, shape, old_s, new_s)
    return dict(shape=shape, old_s=old_s, new_s=new_s, old=old, new=new, rec=rec)


def _link_rejected(ctx, old, new, rec, reason):
    ok, why = keygen.powers_verify_contribution(ctx, old, new, rec)
    assert not ok
    assert reason in why, why


def test_verify_contribution_rejects(gp, link):
    old, new, rec = link["old"], link["new"], link["rec"]
    assert keygen.powers_verify_contribution(gp.ctx, old, new, rec) == (True, "")
    # the record of another contribution
    _, other_rec = keygen.powers_contribute(gp.ctx, old, *link["new_s"])
    assert other_rec != rec                                  # fresh nonces
    assert keygen.powers_verify_contribution(gp.ctx, old, new, other_rec)[0]
    _, foreign = keygen.powers_contribute(gp.ctx, old, *secrets(52))
    _link_rejected(gp.ctx, old, new, foreign, "the tau proof of knowledge does not hold")
    # z + 1, another R
    for j, name in enumerate(NAMES):
        z = int.from_bytes(rec[96 * j + 64:96 * j + 96], "little")
        bad_z = rec[:96 * j + 64] + ((z + 1) % R).to_bytes(32, "little") + rec[96 * j + 96:]
        _link_rejected(gp.ctx, old, new, bad_z, "the %s proof of knowledge does not hold" % name)
        bad_r = rec[:96 * j] + _points(gp.ctx, 1, [99]) + rec[96 * j + 64:]
        _link_rejected(gp.ctx, old, new, bad_r, "the %s proof of knowledge does not hold" % name)
    _link_rejected(gp.ctx, old, new, rec[:64] + R.to_bytes(32, "little") + rec[96:], "the tau proof's z is >= r")
    _link_rejected(gp.ctx, old, new, b"\0" * 64 + rec[64:], "the tau proof's R is the point at infinity")
    # well formed but unlinked: fresh powers of another tau
    fresh = powers(gp.ctx, *secrets(53), *link["shape"])
    assert keygen.powers_verify(gp.ctx, fresh)[0]
    _link_rejected(gp.ctx, old, fresh, rec, "the tau proof of knowledge does not hold")
    # a correct tau link with alpha replaced
    tau = link["old_s"][0] * link["new_s"][0] % R
    alt = dict(new, alpha_tau_g1=_points(gp.ctx, 1, _pows(tau, counts(new)[2], 12345)))
    assert keygen.powers_verify(gp.ctx, alt)[0]
    _link_rejected(gp.ctx, old, alt, rec, "the alpha proof of knowledge does not hold")
    # old and new swapped
    _link_rejected(gp.ctx, new, old, rec, "proof of knowledge does not hold")
    # a valid record over malformed new powers: the full verification still runs
    _link_rejected(gp.ctx, old, _replace(new, "tau_g1", 30, _points(gp.ctx, 1, [3])), rec, "G1 same-ratio check failed")
    # counts that differ are an error, not a verdict
    with pytest.raises(_lib.ZkrError) as e:
        keygen.powers_verify_contribution(gp.ctx, old, dict(new, tau_g1=new["tau_g1"][:-64]), rec)
    assert e.value.code == -1 and "different counts" in str(e.value)


def test_null_secrets(gp, link):
    a, ra = keygen.powers_contribute(gp.ctx, link["old"])
    b, rb = keygen.powers_contribute(gp.ctx, link["old"])
    assert a["tau_g1"] != b["tau_g1"] and a["beta_g2"] != b["beta_g2"] and ra != rb
    for p, r in ((a, ra), (b, rb)):
        assert keygen.powers_verify_contribution(gp.ctx, link["old"], p, r) == (True, "")
    with pytest.raises(ValueError):
        keygen.powers_contribute(gp.ctx, link["old"], tau=5)


# ------------------------------------------------------------------------------------------------ refusals
def _err(fn):
    with pytest.raises(_lib.ZkrError) as e:
        fn()
    assert e.value.code == -1
    return str(e.value)


def test_refusals_before_any_launch(gp, link):
    p = link["old"]
    L = _lib.lib()
    before = L.zkr_ctx_kernel_launches(gp.ctx)
    contrib = lambda q, s=(3, 4, 5): _err(lambda: keygen.powers_contribute(gp.ctx, q, *s))
    assert "tau_g1 has 1 points, 2 needed" in contrib(dict(p, tau_g1=p["tau_g1"][:64]))
    assert "tau_g2 has 1 points, 2 needed" in contrib(dict(p, tau_g2=p["tau_g2"][:128]))
    assert "alpha_tau_g1 has 0 points, 1 needed" in contrib(dict(p, alpha_tau_g1=b""))
    assert "beta_tau_g1 has 0 points, 1 needed" in contrib(dict(p, beta_tau_g1=b""))
    assert "zkr_powers_contribute: tau_g1[7] is not on the curve" in contrib(
        _replace(p, "tau_g1", 7, p["tau_g1"][7 * 64:7 * 64 + 32] + _mont(5)))
    assert "beta_tau_g1[3] has a coordinate >= q" in contrib(_replace(p, "beta_tau_g1", 3, Q.to_bytes(32, "little")))
    assert "alpha_tau_g1[0] is the point at infinity" in contrib(_replace(p, "alpha_tau_g1", 0, b"\0" * 32))
    assert "tau_g2[2] is the point at infinity" in contrib(_replace(p, "tau_g2", 2, b"\0" * 64))
    assert "beta_g2[0] has a coordinate >= q" in contrib(_replace(p, "beta_g2", 0, p["beta_g2"][:96] + (Q + 5).to_bytes(32, "little")))
    assert "tau must be in [1, r)" in contrib(p, (0, 1, 1))
    assert "alpha must be in [1, r)" in contrib(p, (1, R, 1))
    assert "beta must be in [1, r)" in contrib(p, (1, 1, R + 1))
    assert "tau_g2 has 1 points, 2 needed" in _err(lambda: keygen.powers_verify(gp.ctx, dict(p, tau_g2=p["tau_g2"][:128])))
    assert L.zkr_ctx_kernel_launches(gp.ctx) == before
