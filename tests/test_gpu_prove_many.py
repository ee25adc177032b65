"""zkr_prove_many / zkr_msm_many: many witnesses (scalar vectors) of one key (base set) in one pass.

Every batched proof must equal zkr_prove's on the same witness and (r, s), byte for byte, and the committed oracle KATs;
every batched MSM result must equal zkr_msm of its vector, and one size a host-only expectation.  A batch keys proof j's
digits j * nbuckets + |digit| - 1, so a heavy bucket of one proof (the same witness in every slot, all-(r - 1) or all-zero
witnesses) must never leak into another's."""
import base64
import ctypes as C
import gzip
import json
import os
import random

import numpy as np
import pytest

from oracle import binfmt as bf
from oracle import bn254 as bn
from oracle import groth16 as g
from oracle.bn254 import R
from simple_zk_rollups_b200 import _lib, keygen, prover, synth
from helpers import affine_std, pack, pack_g1, pack_g2

pytestmark = pytest.mark.gpu

TOXIC = (0x1234567890ABCDEF1234567890ABCDEF1234567, 0x2222222222222222222222222222222222221,
         0x3333333333333333333333333333333333333331, 0x44444444444444444444444444444444441,
         0x555555555555555555555555555555555555555551)
KATS = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "groth16_kats.json")))


@pytest.fixture(scope="module")
def gp():
    p = prover.Groth16Prover(0)
    yield p
    p.close()


def _variants(w, npub, k, rng):
    """k distinct witnesses of one circuit (public inputs and a few private signals changed: well formed, most of them
    circuit-violating, which the prover must still reproduce exactly) and k distinct (r, s), including r = s = 0."""
    ws, rs = [], []
    for j in range(k):
        wj = list(w)
        if j:
            for i in rng.sample(range(1, len(w)), min(3, len(w) - 1)):
                wj[i] = rng.randrange(R)
        ws.append(wj)
        rs.append((0, 0) if j == 0 else (rng.randrange(R), rng.randrange(R)))
    return ws, rs


def _check_batch(gp, key, ws, rs, handle=None):
    wbins = [bf.binarify_witness(x) for x in ws]
    own = handle is None
    h = handle or gp.create_many(key, len(ws))
    try:
        got = gp.prove_many(h, wbins, rs)
    finally:
        if own:
            h.close()
    assert len(got) == len(ws)
    for j, (wb, (r, s)) in enumerate(zip(wbins, rs)):
        assert got[j] == gp.prove(key, wb, r, s)[0], "proof %d of %d differs from zkr_prove" % (j, len(ws))
    return got


@pytest.mark.parametrize("nc,npub,seed", [(5, 1, 1), (50, 3, 2), (200, 10, 3), (1000, 4, 4)])
def test_prove_many_matches_single_proofs_small(gp, nc, npub, seed):
    r1, w = synth.generate(nc, npub, seed=seed)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    rng = random.Random(seed)
    for k in (1, 2, 3, 17, 64):
        ws, rs = _variants(w, npub, k, rng)
        got = _check_batch(gp, key, ws, rs)
    # the honest witness at r = s = 0 (slot 0) against the oracle, and it verifies
    want, pub = g.gen_proof(pk, w, 0, 0)
    assert got[0] == g.proof_to_bytes(want)
    assert g.verify(vk, g.proof_from_bytes(got[0]), pub)


def _kat_pk(v):
    return gzip.decompress(base64.b64decode(v["pk_bin_gz_b64"]))


@pytest.mark.parametrize("vi", [0, 1])
def test_prove_many_reproduces_kats(gp, vi):
    """The committed oracle vectors, honest and circuit-violating, all in one batch."""
    v = KATS["vectors"][vi]
    key = gp.load_key(_kat_pk(v))
    w = [int(x) for x in v["witness"]]
    bad = list(w)
    bad[v["invalid_witness"]["index"]] = int(v["invalid_witness"]["witness_value"])
    ws = [w] * len(v["proofs"]) + [bad]
    rs = [(int(p["r"]), int(p["s"])) for p in v["proofs"]] + [(int(v["invalid_witness"]["r"]), int(v["invalid_witness"]["s"]))]
    want = [p["proof_hex"] for p in v["proofs"]] + [v["invalid_witness"]["proof_hex"]]
    h = gp.create_many(key, len(ws))
    got = gp.prove_many(h, [bf.binarify_witness(x) for x in ws], rs)
    h.close()
    assert [x.hex() for x in got] == want


@pytest.fixture(scope="module")
def shapes(gp):
    """withdraw and tx shapes: key, witness (GPU setup, as test_prove_full_size)."""
    out = {}
    for shape in ("withdraw", "tx"):
        nc, npub = synth.SHAPES[shape]
        r1, w = synth.generate(nc, npub, seed=11)
        pk_bin, vk = keygen.synth_setup(gp.ctx, r1, TOXIC)
        out[shape] = (gp.load_key(pk_bin), w, npub, vk)
    return out


@pytest.mark.parametrize("shape,ks", [("withdraw", (1, 2, 3, 17, 64, 256)), ("tx", (1, 2, 3, 17, 64))])
def test_prove_many_full_shapes(gp, shapes, shape, ks):
    key, w, npub, vk = shapes[shape]
    rng = random.Random(len(shape))
    for k in ks:
        ws, rs = _variants(w, npub, k, rng)
        got = _check_batch(gp, key, ws, rs)
    # slot 0 is the honest witness: the proof verifies
    vkey = gp.load_vkey(vk["bin"])
    assert gp.verify(vkey, got[0], w[1:npub + 1])


def test_prove_many_adversarial_batches(gp):
    r1, w = synth.generate(300, 4, seed=12)
    pk, _, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    n = len(w)
    same = [list(w)] * 9
    top = [1] + [R - 1] * (n - 1)
    zero = [1] + [0] * (n - 1)
    violating = list(w)
    violating[10] = (violating[10] + 12345) % R
    rng = random.Random(3)
    rs9 = [(rng.randrange(R), rng.randrange(R)) for _ in range(9)]
    _check_batch(gp, key, same, rs9)                                  # one heavy bucket per window in every proof
    _check_batch(gp, key, [top] * 5, rs9[:5])
    _check_batch(gp, key, [zero] * 5, [(0, 0)] + rs9[:4])             # all-zero digits but w0: near-empty buckets
    got = _check_batch(gp, key, [violating], [(7, 9)])
    assert got[0] == g.proof_to_bytes(g.gen_proof(pk, violating, 7, 9, h_method=g.calc_h_websnark)[0])
    mixed = [w, top, zero, violating, w, top, zero, violating, w]
    _check_batch(gp, key, mixed, rs9)


def test_prove_many_workspace_reuse_and_errors(gp):
    r1, w = synth.generate(150, 3, seed=13)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    rng = random.Random(13)
    ws64, rs64 = _variants(w, 3, 64, rng)
    ws3, rs3 = ws64[:3], rs64[:3]
    h = gp.create_many(key, 64)
    info = h.info()
    assert info["max_proofs"] == 64 and info["device_bytes"] > 0
    a = _check_batch(gp, key, ws64, rs64, h)
    b = _check_batch(gp, key, ws3, rs3, h)
    c = _check_batch(gp, key, ws64, rs64, h)
    assert a == c and b == a[:3]
    # a bad value in proof j: ZKR_E_WITNESS_RANGE naming j, then the workspace is clean
    bad = [list(x) for x in ws3]
    bad[2][5] = R
    with pytest.raises(_lib.ZkrError) as ei:
        gp.prove_many(h, [bf.binarify_witness(x) for x in bad], rs3)
    assert ei.value.code == -3 and "proof 2" in str(ei.value)
    bad = [list(x) for x in ws3]
    bad[1][0] = 2
    with pytest.raises(_lib.ZkrError) as ei:
        gp.prove_many(h, [bf.binarify_witness(x) for x in bad], rs3)
    assert ei.value.code == -3 and "proof 1" in str(ei.value)
    assert _check_batch(gp, key, ws3, rs3, h) == b
    wb = [bf.binarify_witness(x) for x in ws3]
    L = gp.L
    out = np.zeros(256 * 70, dtype=np.uint8)
    flat = np.frombuffer(b"".join(wb), dtype=np.uint8)
    for n_proofs in (0, 65):                                          # n_proofs out of range
        assert L.zkr_prove_many(gp.ctx, h.h, _lib.buf_ptr(flat), len(w), n_proofs, None, _lib.buf_ptr(out)) == -1
    assert L.zkr_prove_many(gp.ctx, h.h, _lib.buf_ptr(flat), len(w) - 1, 3, None, _lib.buf_ptr(out)) == -1
    for bad_rs in ([(1, 2), (R, 0), (3, 4)], [(1, 2), (3, 4), (5, R)]):
        with pytest.raises(_lib.ZkrError) as ei:
            gp.prove_many(h, wb, bad_rs)
        assert ei.value.code == -1
    # rs = NULL: fresh CSPRNG pairs, pairwise distinct proofs that verify
    honest = [bf.binarify_witness(w)] * 4
    rnd = gp.prove_many(h, honest)
    assert len(set(rnd)) == 4
    assert all(g.verify(vk, g.proof_from_bytes(p), w[1:4]) for p in rnd)
    h.close()


def test_prove_many_launches_do_not_grow_with_k(gp):
    r1, w = synth.generate(400, 3, seed=14)
    pk, _, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    h = gp.create_many(key, 64)
    wb = bf.binarify_witness(w)
    gp.prove_many(h, [wb], [(1, 2)])                  # builds this size's cached NTT tables (cold-path launches)
    counts = []
    for k in (1, 64, 1):
        before = gp.kernel_launches()
        gp.prove_many(h, [wb] * k, [(1, 2)] * k)
        counts.append(gp.kernel_launches() - before)
    h.close()
    assert counts[0] == counts[1] == counts[2], counts


def test_prove_many_rejects_sharded_key(gp):
    r1, w = synth.generate(100, 3, seed=15)
    pk, _, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key_sharded(bf.binarify_proving_key(pk), 0, 2)
    with pytest.raises(_lib.ZkrError) as ei:
        gp.create_many(key, 4)
    assert ei.value.code == -8


# ------------------------------------------------------------------------------------------------ standalone batched MSM
def _load(gp, group, pts, c):
    arr = pack_g1(pts) if group == 1 else pack_g2(pts)
    h = C.c_void_p()
    _lib.check(gp.L.zkr_bases_load(gp.ctx, group, _lib.buf_ptr(arr), len(pts), c, C.byref(h)))
    return h


def _msm(gp, group, h, scalars):
    out = np.zeros(64 if group == 1 else 128, dtype=np.uint8)
    sc = pack(scalars)
    _lib.check(gp.L.zkr_msm(gp.ctx, h, _lib.buf_ptr(sc), len(scalars), 0, _lib.buf_ptr(out)))
    return out.tobytes()


@pytest.mark.parametrize("c", [0, 21])                # c = 0: chosen from n (the gather); 21: the boundary levels
@pytest.mark.parametrize("group", [1, 2])
def test_msm_many_matches_single_msms(gp, group, c):
    n = 700 if group == 1 else 300
    rng = random.Random(group * 100 + c)
    exps = [rng.randrange(1, R) for _ in range(n)]
    exps[3] = 0                                       # an infinity base
    pts = bn.fixed_base(group).mul_many(exps)
    h = _load(gp, group, pts, c)
    base_vecs = [[0] * n, [R - 1] * n, [rng.randrange(R) for _ in range(n)], [1] * n]
    for k in (1, 2, 5, 64):
        vecs = [base_vecs[j % 4] if j < 8 else [rng.randrange(R) for _ in range(n)] for j in range(k)]
        if k > 2:
            vecs[-1] = vecs[2]                        # a repeated vector
        got = gp.msm_many(h, b"".join(pack(v).tobytes() for v in vecs), n, k, group)
        for j, v in enumerate(vecs):
            assert got[j] == _msm(gp, group, h, v), (k, j)
        if k >= 1:
            assert got[0] == bytes(64 if group == 1 else 128)          # the all-zero vector: infinity
    gp.L.zkr_bases_free(h)


@pytest.mark.parametrize("group", [1, 2])
def test_msm_many_host_expectation_and_range_error(gp, group):
    """P_i = e_i G, result j = (sum_i k_ji e_i mod r) G, computed on the host (as test_gpu_msm_plans.py)."""
    n, k = 257, 9
    rng = random.Random(7 + group)
    exps = [rng.randrange(R) for _ in range(n)]
    pts = bn.fixed_base(group).mul_many(exps)
    h = _load(gp, group, pts, 0)
    vecs = [[rng.randrange(R) for _ in range(n)] for _ in range(k)]
    got = gp.msm_many(h, b"".join(pack(v).tobytes() for v in vecs), n, k, group)
    want = bn.fixed_base(group).mul_many([sum(a * e for a, e in zip(v, exps)) % R for v in vecs])
    ob = 64 if group == 1 else 128
    for j in range(k):
        assert affine_std(group, np.frombuffer(got[j], dtype=np.uint8)) == want[j], j
    vecs[4][10] = R
    with pytest.raises(_lib.ZkrError) as ei:
        gp.msm_many(h, b"".join(pack(v).tobytes() for v in vecs), n, k, group)
    assert ei.value.code == -3 and "vector 4" in str(ei.value)
    vecs[4][10] = 5
    got2 = gp.msm_many(h, b"".join(pack(v).tobytes() for v in vecs[:3]), n, 3, group)
    assert got2 == got[:3] and all(len(x) == ob for x in got2)
    gp.L.zkr_bases_free(h)
