"""Setup from powers of tau and phase-2 delta contributions (csrc/ceremony.cu, zkr.h "setup from a powers-of-tau
ceremony").

The setup is deterministic in its secrets, so every path is checked byte for byte against zkr_synth_setup for the
matching toxic waste: setup_from_powers(powers(tau, alpha, beta)) == synth_setup(tau, alpha, beta, 1, 1), and
contribute(., d) == synth_setup(tau, alpha, beta, 1, d).  Synthetic powers come from scalars computed with Python
ints and turned into points by zkr_synth_points.  The contribution record is re-derived with hashlib and checked on
the oracle's integer curve arithmetic."""
import hashlib
import random
import struct

import numpy as np
import pytest

from oracle import bn254 as bn
from simple_zk_rollups_b200 import _lib, keygen, prover, synth

R, Q = bn.R, bn.Q
RINV_Q = pow(1 << 256, -1, Q)
SECTIONS = ("polsA", "polsB", "A", "B1", "B2", "C", "H")

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


def powers(ctx, m, tau, alpha, beta, n_g1=None):
    """Phase-1 points of a ceremony of size m: tau_g1 has n_g1 (default 2m) points, the others m."""
    n_g1 = 2 * m if n_g1 is None else n_g1
    return {"tau_g1": _points(ctx, 1, _pows(tau, n_g1)), "tau_g2": _points(ctx, 2, _pows(tau, m)),
            "alpha_tau_g1": _points(ctx, 1, _pows(tau, m, alpha)), "beta_tau_g1": _points(ctx, 1, _pows(tau, m, beta)),
            "beta_g2": _points(ctx, 2, [beta])}


def sections(pk):
    pk = bytes(pk)
    hdr = struct.unpack_from("<10I", pk)
    ptrs = list(hdr[3:]) + [len(pk)]
    out = {"header": pk[:ptrs[0]]}
    for i, name in enumerate(SECTIONS):
        out[name] = pk[ptrs[i]:ptrs[i + 1]]
    return out


def assert_same_key(pk1, vk1, pk2, vk2):
    s1, s2 = sections(pk1), sections(pk2)
    for name in s1:
        if s1[name] != s2[name]:
            size = 128 if name == "B2" else 64
            first = next(i for i in range(len(s1[name])) if s1[name][i] != s2[name][i])
            pytest.fail("section %s differs first at point %d" % (name, first // size))
    assert bytes(vk1["bin"]) == bytes(vk2["bin"])
    assert bytes(pk1) == bytes(pk2)


def secrets(seed):
    rng = random.Random(seed)
    return [rng.randrange(1, R) for _ in range(3)]


def _shape(log_m, over):
    """synth.py shape with n > m (nConstraints + nPublic + 1 = m) or n < m (= m/2 + 1, no free signals)."""
    m = 1 << log_m
    l = min(5, max(0, m // 4)) if over else max(1, min(5, m // 8))
    if over:
        return synth.generate(m - l - 1, l, seed=log_m)[0]
    return synth.generate(m // 2 - l, l, seed=100 + log_m, n_free=0)[0]


@pytest.mark.parametrize("log_m,over", [(k, True) for k in range(1, 13)] + [(k, False) for k in range(2, 13)])
def test_from_powers_matches_synth_setup(gp, log_m, over):
    r1 = _shape(log_m, over)
    bits, m = r1.domain()
    assert m == 1 << log_m and (r1.nVars > m) == over
    tau, alpha, beta = secrets(log_m * 2 + over)
    got = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, m, tau, alpha, beta))
    want = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
    assert_same_key(*got, *want)


def test_shapes_have_empty_columns():
    """The shapes above include signals with empty A and B columns (infinity outputs)."""
    for log_m, over in ((4, True), (8, False), (12, True)):
        ptr = _shape(log_m, over).csc(with_inputs=True)["A"][0].astype(np.int64)
        assert (np.diff(ptr) == 0).any()


def test_from_powers_heavy_column(gp):
    """Signal 1 in every row of A and C (16383 entries: several levels of the segmented sum), m = 2^14."""
    r1, _ = synth.generate(16383 - 3, 2, seed=7)
    rng = np.random.default_rng(7)
    for mat in ("A", "C"):
        sig, row, cid = r1.mats[mat]
        have = set(row[sig == 1].tolist())
        extra = np.array(sorted(set(range(r1.nConstraints)) - have), dtype=np.uint32)
        sig2 = np.concatenate([sig, np.ones(extra.size, dtype=np.uint32)])
        row2 = np.concatenate([row, extra])
        cid2 = np.concatenate([cid, rng.integers(0, len(r1.pool), extra.size).astype(np.uint32)])
        o = np.lexsort((row2, sig2))
        r1.mats[mat] = (sig2[o], row2[o], cid2[o])
    ptr = r1.csc(with_inputs=True)["A"][0].astype(np.int64)
    assert np.diff(ptr).max() >= 10 ** 4
    bits, m = r1.domain()
    assert m == 1 << 14
    tau, alpha, beta = secrets(14)
    got = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, m, tau, alpha, beta))
    want = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
    assert_same_key(*got, *want)


@pytest.mark.parametrize("shape", ["tx", "tx_2p20"])
def test_from_powers_rollup_shapes(gp, shape):
    r1, _ = synth.generate(*synth.SHAPES[shape])
    bits, m = r1.domain()
    tau, alpha, beta = secrets(bits)
    got = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, m, tau, alpha, beta))
    want = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
    assert_same_key(*got, *want)


def test_larger_ceremony_and_exact_size_ceremony(gp):
    """A ceremony of size 4m gives the same bytes.  One of size m (2m - 1 G1 powers) differs only in H_(m-1), which is
    infinity, and proves byte-identically: h_(m-1) = 0 for every satisfying witness."""
    r1, w = synth.generate(200, 5, seed=11)
    bits, m = r1.domain()
    tau, alpha, beta = secrets(21)
    want = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
    big = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, 4 * m, tau, alpha, beta))
    assert_same_key(*big, *want)
    exact_pk, exact_vk = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, m, tau, alpha, beta, n_g1=2 * m - 1))
    s1, s2 = sections(exact_pk), sections(want[0])
    for name in s1:
        if name != "H":
            assert s1[name] == s2[name], name
    assert s1["H"][:-64] == s2["H"][:-64]
    assert s1["H"][-64:] == b"\0" * 32 + (bn.MONT_R % Q).to_bytes(32, "little")
    assert bytes(exact_vk["bin"]) == bytes(want[1]["bin"])
    d = 987654321987654321
    ka = keygen.contribute(gp.ctx, exact_pk, exact_vk, d)
    kb = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, d))
    pa, _ = gp.prove(gp.load_key(ka[0]), synth.witness_bytes(w), 3, 4)
    pb, _ = gp.prove(gp.load_key(kb[0]), synth.witness_bytes(w), 3, 4)
    assert pa == pb
    assert gp.verify(gp.load_vkey(ka[1]["bin"]), pa, w[1:6])
    # the infinity H_(m-1) must stay in the encoding a contribution writes, (0, R mod q)
    assert keygen.verify_contribution(gp.ctx, exact_pk, exact_vk, *ka)
    odd = np.frombuffer(bytes(ka[0]), dtype=np.uint8).copy()
    odd[-32:] = np.frombuffer((2 * bn.MONT_R % Q).to_bytes(32, "little"), dtype=np.uint8)
    assert not keygen.verify_contribution(gp.ctx, exact_pk, exact_vk, odd, ka[1], ka[2])


# ------------------------------------------------------------------------------------------------ contributions
@pytest.fixture(scope="module")
def small(gp):
    r1, w = synth.generate(300, 4, seed=5)
    bits, m = r1.domain()
    tau, alpha, beta = secrets(99)
    pk, vk = keygen.setup_from_powers(gp.ctx, r1, powers(gp.ctx, m, tau, alpha, beta))
    return dict(r1=r1, w=w, toxic=(tau, alpha, beta), pk=pk, vk=vk)


def test_contribution_is_byte_identical(gp, small):
    tau, alpha, beta = small["toxic"]
    d1, d2 = 1234567890123456789012345678901234567890 % R, R - 2
    pk1, vk1, rec1 = keygen.contribute(gp.ctx, small["pk"], small["vk"], d1)
    assert_same_key(pk1, vk1, *keygen.synth_setup(gp.ctx, small["r1"], (tau, alpha, beta, 1, d1)))
    pk2, vk2, rec2 = keygen.contribute(gp.ctx, pk1, vk1, d2)
    assert_same_key(pk2, vk2, *keygen.synth_setup(gp.ctx, small["r1"], (tau, alpha, beta, 1, d1 * d2 % R)))
    assert keygen.verify_contribution(gp.ctx, small["pk"], small["vk"], pk1, vk1, rec1)
    assert keygen.verify_contribution(gp.ctx, pk1, vk1, pk2, vk2, rec2)


def test_contribution_at_tx_shape_is_byte_identical(gp):
    r1, _ = synth.generate(*synth.SHAPES["tx"])
    tau, alpha, beta = secrets(3)
    d = 31337
    pk, vk = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
    pk1, vk1, rec = keygen.contribute(gp.ctx, pk, vk, d)
    assert_same_key(pk1, vk1, *keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, d)))
    assert keygen.verify_contribution(gp.ctx, pk, vk, pk1, vk1, rec)


def test_proofs_with_contributed_key(gp, small):
    tau, alpha, beta = small["toxic"]
    w = small["w"]
    d = 5 ** 100 % R
    pk1, vk1, _ = keygen.contribute(gp.ctx, small["pk"], small["vk"], d)
    ref_pk, ref_vk = keygen.synth_setup(gp.ctx, small["r1"], (tau, alpha, beta, 1, d))
    pa, _ = gp.prove(gp.load_key(pk1), synth.witness_bytes(w), 11, 12)
    pb, _ = gp.prove(gp.load_key(ref_pk), synth.witness_bytes(w), 11, 12)
    assert pa == pb
    assert gp.verify(gp.load_vkey(vk1["bin"]), pa, w[1:5])
    assert not gp.verify(gp.load_vkey(small["vk"]["bin"]), pa, w[1:5])


def _g1_mont(b):
    x = int.from_bytes(b[:32], "little") * RINV_Q % Q
    y = int.from_bytes(b[32:64], "little") * RINV_Q % Q
    return None if x == 0 else (x, y)


def _delta1(pk):
    return bytes(pk[168:232])


def test_record_pinned_from_outside(gp, small):
    """c = SHA-256("zkr-phase2-delta" | delta1_old | delta1_new | R) mod r and z delta1_old = R + c delta1_new on
    oracle integers; with a known delta', z - c delta' = k and R = k delta1_old."""
    d = 424242424242
    pk1, vk1, rec = keygen.contribute(gp.ctx, small["pk"], small["vk"], d)
    old, new, Rb = _delta1(small["pk"]), _delta1(pk1), rec[:64]
    z = int.from_bytes(rec[64:], "little")
    assert z < R
    c = int.from_bytes(hashlib.sha256(b"zkr-phase2-delta" + old + new + Rb).digest(), "little") % R
    P_old, P_new, P_R = _g1_mont(old), _g1_mont(new), _g1_mont(Rb)
    assert P_new == bn.G1.mul(P_old, d)
    assert bn.G1.mul(P_old, z) == bn.G1.add(P_R, bn.G1.mul(P_new, c))
    assert P_R == bn.G1.mul(P_old, (z - c * d) % R)


def test_verifier_accepts_random_contributions(gp, small):
    a = keygen.contribute(gp.ctx, small["pk"], small["vk"])
    b = keygen.contribute(gp.ctx, small["pk"], small["vk"])
    assert bytes(a[0]) != bytes(b[0]) and a[2] != b[2]
    assert _delta1(a[0]) != _delta1(b[0])
    for pk1, vk1, rec in (a, b):
        assert keygen.verify_contribution(gp.ctx, small["pk"], small["vk"], pk1, vk1, rec)
    c = keygen.contribute(gp.ctx, a[0], a[1])
    assert keygen.verify_contribution(gp.ctx, a[0], a[1], c[0], c[1], c[2])


def _mont_point(ctx, k):
    return _points(ctx, 1, [k])


def test_verifier_rejects(gp, small):
    pk0, vk0 = small["pk"], small["vk"]
    pk1, vk1, rec = keygen.contribute(gp.ctx, pk0, vk0, 777)
    other = keygen.contribute(gp.ctx, pk0, vk0, 778)
    sec = sections(pk1)
    hdr = struct.unpack_from("<10I", bytes(pk1))
    pC, pH = hdr[8], hdr[9]
    ok = lambda pk=pk1, vk=vk1, r=rec, opk=pk0, ovk=vk0: keygen.verify_contribution(gp.ctx, opk, ovk, pk, vk, r)
    assert ok()

    def patched(buf, off, data):
        b = np.frombuffer(bytes(buf), dtype=np.uint8).copy()
        b[off:off + len(data)] = np.frombuffer(data, dtype=np.uint8)
        return b

    # one C point changed (to another valid point), the last H point changed, H scaled by another scalar
    assert len(sec["C"]) >= 64
    assert not ok(pk=patched(pk1, pC, _mont_point(gp.ctx, 12345)))
    assert not ok(pk=patched(pk1, len(pk1) - 64, _mont_point(gp.ctx, 54321)))
    scaled = keygen.contribute(gp.ctx, pk0, vk0, 779)[0]
    assert not ok(pk=patched(pk1, pH, bytes(scaled[pH:])))
    # delta2 not matching delta1 (in both the key and the vk)
    d2 = bytes(other[0][360:488])
    assert not ok(pk=patched(pk1, 360, d2), vk={"bin": bytes(patched(vk1["bin"], 448, d2))})
    # z or R altered, a record of another contribution
    bad_z = rec[:64] + ((int.from_bytes(rec[64:], "little") + 1) % R).to_bytes(32, "little")
    assert not ok(r=bad_z)
    assert not ok(r=_mont_point(gp.ctx, 99) + rec[64:])
    assert not ok(r=other[2])
    # one byte changed in A, B1, B2, IC, the header, polsA
    for off in (hdr[5] + 3, hdr[6] + 70, hdr[7] + 5, hdr[3] + 9, 4, hdr[3] + 1):
        b = np.array(pk1, dtype=np.uint8, copy=True)
        b[off] ^= 1
        assert not ok(pk=b), off
    ic = bytearray(vk1["bin"])
    ic[576 + 64 + 1] ^= 1
    assert not ok(vk={"bin": bytes(ic)})
    # old and new swapped
    assert not ok(pk=pk0, vk=vk0, opk=pk1, ovk=vk1)
    # a malformed layout is an error, not a verdict
    with pytest.raises(_lib.ZkrError) as e:
        keygen.verify_contribution(gp.ctx, pk0[:-64], vk0, pk1[:-64], vk1, rec)
    assert e.value.code == -1


def _err(fn):
    with pytest.raises(_lib.ZkrError) as e:
        fn()
    assert e.value.code == -1
    return str(e.value)


def test_bad_powers_are_refused_before_any_launch(gp):
    r1, _ = synth.generate(100, 3, seed=2)
    bits, m = r1.domain()
    pw = powers(gp.ctx, m, *secrets(5))
    L = _lib.lib()
    before = L.zkr_ctx_kernel_launches(gp.ctx)

    def run(name, data):
        p = dict(pw)
        p[name] = data
        return _err(lambda: keygen.setup_from_powers(gp.ctx, r1, p))

    assert "tau_g1 has %d points, %d needed" % (2 * m - 2, 2 * m - 1) in run("tau_g1", pw["tau_g1"][:64 * (2 * m - 2)])
    assert "tau_g2 has %d points" % (m - 1) in run("tau_g2", pw["tau_g2"][:-128])
    assert "alpha_tau_g1 has" in run("alpha_tau_g1", pw["alpha_tau_g1"][:-64])
    assert "beta_tau_g1 has" in run("beta_tau_g1", b"")

    def patch(name, idx, size, data, at=0):
        b = bytearray(pw[name])
        b[idx * size + at:idx * size + at + len(data)] = data
        return bytes(b)

    assert "tau_g1[7] is not on the curve" in run("tau_g1", patch("tau_g1", 7, 64, b"\x01", at=32))
    # tau^(2m-1) is read when given (it makes H_(m-1)), so it is checked too
    assert "tau_g1[%d] is not on the curve" % (2 * m - 1) in run("tau_g1", patch("tau_g1", 2 * m - 1, 64, b"\x01", at=32))
    assert "tau_g1[%d] is the point at infinity" % (2 * m - 1) in run("tau_g1", patch("tau_g1", 2 * m - 1, 64, b"\0" * 32))
    assert "beta_tau_g1[3] has a coordinate >= q" in run("beta_tau_g1", patch("beta_tau_g1", 3, 64, Q.to_bytes(32, "little")))
    assert "alpha_tau_g1[0] is the point at infinity" in run("alpha_tau_g1", patch("alpha_tau_g1", 0, 64, b"\0" * 32))
    assert "tau_g2[5] is not on the curve" in run("tau_g2", patch("tau_g2", 5, 128, b"\x02", at=64))
    assert "tau_g2[2] is the point at infinity" in run("tau_g2", patch("tau_g2", 2, 128, b"\0" * 64))
    assert "beta_g2[0] has a coordinate >= q" in run("beta_g2", patch("beta_g2", 0, 128, (Q + 5).to_bytes(32, "little"), at=96))
    assert L.zkr_ctx_kernel_launches(gp.ctx) == before
