"""GPU parity for the whole hot path: zkr_prove vs the oracle's gen_proof, byte for byte with fixed (r, s);
the proof must verify under the restated on-chain predicate (TxVerifier.sol:258-276) and a tampered
public input must fail (contracts/__tests__/withdrawverifier.test.ts:42-68)."""
import random
import time

import numpy as np
import pytest

from oracle import binfmt as bf
from oracle import groth16 as g
from oracle.bn254 import R
from simple_zk_rollups_b200 import _lib, binarify, keygen, prover, synth

pytestmark = pytest.mark.gpu

TOXIC = (0x1234567890ABCDEF1234567890ABCDEF1234567, 0x2222222222222222222222222222222222221,
         0x3333333333333333333333333333333333333331, 0x44444444444444444444444444444444441,
         0x555555555555555555555555555555555555555551)


@pytest.fixture(scope="module")
def gp():
    p = prover.Groth16Prover(0)
    yield p
    p.close()


@pytest.mark.parametrize("nc,npub,seed", [(5, 1, 1), (50, 3, 2), (200, 10, 3), (1000, 4, 4)])
def test_prove_bit_exact_small(gp, nc, npub, seed):
    r1, w = synth.generate(nc, npub, seed=seed)
    pk, vk, sec = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    info = gp.key_info(key)
    assert (info["nVars"], info["nPublic"], info["domainSize"]) == (pk["nVars"], pk["nPublic"], pk["domainSize"])
    wbin = bf.binarify_witness(w)
    rng = random.Random(seed)
    for r, s in ((0, 0), (1, 0), (0, 1), (rng.randrange(R), rng.randrange(R)), (R - 1, R - 1)):
        got, stats = gp.prove(key, wbin, r, s)
        want, pub = g.gen_proof(pk, w, r, s)
        assert got == g.proof_to_bytes(want), "proof bytes differ at (r,s)=(%d,%d)" % (r, s)
        assert stats["kernel_launches"] > 0
    proof = g.proof_from_bytes(got)
    assert g.verify(vk, proof, pub)
    bad = list(pub)
    bad[0] = (bad[0] + 1) % R
    assert not g.verify(vk, proof, bad)
    assert g.exponent_check(pk, sec, w, proof, R - 1, R - 1)


def test_prove_rejects_bad_inputs(gp):
    r1, w = synth.generate(20, 2, seed=9)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    w2 = list(w)
    w2[5] = R                                   # out of range, must not be silently reduced
    with pytest.raises(_lib.ZkrError) as ei:
        gp.prove(key, bf.binarify_witness(w2))
    assert ei.value.code == -3
    w3 = list(w)
    w3[0] = 2                                   # witness[0] must be the constant 1
    with pytest.raises(_lib.ZkrError) as ei:
        gp.prove(key, bf.binarify_witness(w3))
    assert ei.value.code == -3
    with pytest.raises(_lib.ZkrError):          # wrong length
        gp.prove(key, bf.binarify_witness(w[:-1]))
    with pytest.raises(_lib.ZkrError) as ei:    # blinding scalar out of range
        gp.prove(key, bf.binarify_witness(w), r=R)
    assert ei.value.code == -3
    # still healthy afterwards
    got, _ = gp.prove(key, bf.binarify_witness(w), 3, 4)
    assert got == g.proof_to_bytes(g.gen_proof(pk, w, 3, 4)[0])
    # malformed keys
    good = bf.binarify_proving_key(pk)
    for bad in (good[:100], good[:-1], b"\xff" * 40 + good[40:]):
        with pytest.raises(_lib.ZkrError) as ei:
            gp.load_key(bad)
        assert ei.value.code == -2


def test_invalid_witness_matches_websnark_h(gp):
    """websnark never reads polsC: for a witness violating A.B = C its H is still the upper half of A.B;
    the GPU path must reproduce that (oracle calc_h_websnark), even though the proof will not verify."""
    r1, w = synth.generate(60, 2, seed=5)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    w2 = list(w)
    w2[10] = (w2[10] + 12345) % R
    got, _ = gp.prove(key, bf.binarify_witness(w2), 7, 9)
    want, pub = g.gen_proof(pk, w2, 7, 9, h_method=g.calc_h_websnark)
    assert got == g.proof_to_bytes(want)
    assert not g.verify(vk, g.proof_from_bytes(got), pub)


def test_gpu_setup_matches_oracle_setup(gp):
    """zkr_synth_setup + host assembly == binarifyProvingKey(oracle setup) byte for byte; same vk."""
    r1, w = synth.generate(120, 5, seed=6)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    pk_bin, vk_gpu = keygen.synth_setup(gp.ctx, r1, TOXIC)
    ref = bf.binarify_proving_key(pk)
    assert pk_bin.tobytes() == ref
    assert pk_bin.tobytes() == binarify.binarifyProvingKey(bf.pk_to_json(pk))
    for k in ("vk_alfa_1", "vk_beta_2", "vk_gamma_2", "vk_delta_2", "IC"):
        assert vk_gpu[k] == vk[k], k


def test_api_mirror(gp):
    """createProofGenerator / genProof keep the reference's shapes (common.ts:40-51)."""
    r1, w = synth.generate(30, 3, seed=7)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    pkj, vkj = bf.pk_to_json(pk), bf.vk_to_json(vk)

    def calc(name, inputs):
        assert name == "tx.circom"
        return w, 3

    def is_valid(vkey, proof, pub):
        return g.verify(bf.vk_from_json(vkey), bf.proof_from_json(proof), [int(x) for x in pub])

    gen = prover.createProofGenerator(pkj, vkj, "tx.circom", calc, is_valid, prover=gp)
    out = gen({"any": 1})
    assert set(out) == {"proof", "solidityProof"}
    sp = out["solidityProof"]
    assert len(sp["a"]) == 2 and len(sp["c"]) == 2 and len(sp["b"]) == 2 and len(sp["inputs"]) == 3
    assert sp["b"][0] == list(reversed(out["proof"]["pi_b"][0]))
    assert out["proof"]["pi_a"][2] == "1" and out["proof"]["pi_b"][2] == ["1", "0"]
    res = prover.genProof(pkj, w, 0, 0, prover=gp)
    assert res["publicSignals"] == [str(x) for x in w[1:4]]
    want, _ = g.gen_proof(pk, w, 0, 0)
    assert bf.proof_from_json(res["proof"]) == want
    # a generator whose verifier says no raises like common.ts:36-38
    gen_bad = prover.createProofGenerator(pkj, vkj, "tx.circom", calc, lambda *a: False, prover=gp)
    with pytest.raises(RuntimeError, match="Invalid proof generated"):
        gen_bad({})


def test_prove_from_json_text(gp):
    """SURVEY 8(f) rank 1: proving_key.json / witness.json TEXT -> native ingestion -> resident key -> proof,
    identical to the proof from the binarified key, in the reference's genTxVerifierProof shape."""
    import json
    r1, w = synth.generate(90, 4, seed=21)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    text = json.dumps(bf.pk_to_json(pk), indent=1)
    key = gp.load_key_json(text)
    info = gp.key_info(key)
    assert (info["nVars"], info["nPublic"], info["domainSize"]) == (pk["nVars"], pk["nPublic"], pk["domainSize"])
    wbin = binarify.binarifyWitnessJson(json.dumps([str(x) for x in w]))
    assert wbin == bf.binarify_witness(w)
    got, _ = gp.prove(key, wbin, 11, 13)
    want, pub = g.gen_proof(pk, w, 11, 13)
    assert got == g.proof_to_bytes(want)
    assert g.verify(vk, g.proof_from_bytes(got), pub)
    with pytest.raises(_lib.ZkrError) as ei:
        gp.load_key_json(text[:-20])
    assert ei.value.code == -2


def test_bind_circuit_from_build_directory(gp, tmp_path):
    """tx.ts / withdraw.ts shape: keys come from prover/build/<name>{Proving,Verifying}Key.json files; the generator
    parses them natively once, proves, self-checks with zkr_verify and formats the Solidity call data."""
    import json
    r1, w = synth.generate(70, 3, seed=17)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    (tmp_path / "withdrawProvingKey.json").write_text(json.dumps(bf.pk_to_json(pk)))
    (tmp_path / "withdrawVerifyingKey.json").write_text(json.dumps(bf.vk_to_json(vk)))
    seen = {}

    def calc(name, inputs):
        seen["name"] = name
        return w, 3

    gen = prover.bindCircuit(str(tmp_path), "withdraw", calc, prover=gp)
    out = gen({"x": 1}, r=21, s=22)
    assert seen["name"] == "withdraw.circom"
    assert bf.proof_from_json(out["proof"]) == g.gen_proof(pk, w, 21, 22)[0]
    assert out["solidityProof"]["inputs"] == [str(x) for x in w[1:4]]
    assert out["solidityProof"]["b"][0] == [out["proof"]["pi_b"][0][1], out["proof"]["pi_b"][0][0]]


def test_prove_batch_round_robin(gp):
    """zkr_prove_batch over two contexts (two GPUs when present, else two contexts on device 0): every proof of the
    batch equals the oracle's for its own witness and (r, s), in input order; a bad witness fails the call."""
    import torch
    dev2 = 1 if torch.cuda.device_count() > 1 else 0
    gp2 = prover.Groth16Prover(dev2)
    try:
        r1, w = synth.generate(150, 3, seed=31)
        pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
        pk_bin = bf.binarify_proving_key(pk)
        keys = [gp.load_key(pk_bin), gp2.load_key(pk_bin)]
        wits, rs = [], []
        rng = random.Random(8)
        for i in range(5):
            wi = list(w)
            if i % 2:                      # distinct (well-formed, circuit-violating) witnesses: websnark's H semantics
                wi[7 + i] = (wi[7 + i] + 1000 + i) % R
            wits.append(wi)
            rs.append((rng.randrange(R), rng.randrange(R)))
        proofs = prover.prove_batch([gp, gp2], keys, [bf.binarify_witness(x) for x in wits], rs)
        assert len(proofs) == 5
        for p, wi, (r, s) in zip(proofs, wits, rs):
            assert p == g.proof_to_bytes(g.gen_proof(pk, wi, r, s, h_method=g.calc_h_websnark)[0])
        assert prover.prove_batch([gp, gp2], keys, []) == []
        bad = list(w)
        bad[3] = R
        with pytest.raises(_lib.ZkrError):
            prover.prove_batch([gp, gp2], keys, [bf.binarify_witness(w), bf.binarify_witness(bad)])
    finally:
        gp2.close()


@pytest.mark.parametrize("shape", ["withdraw", "tx", "tx_2p20", "tx_2p22"])
def test_prove_full_size(gp, shape):
    """BASELINE configs[0..1] and the per-GPU unit of configs[4] at full size: GPU setup -> prove -> toxic-waste
    exponent check (no MSM / NTT code shared with the GPU path) -> pairing verification -> tamper-negative ->
    determinism.  The exponent sums are independent of (r, s) and computed once per circuit: on Python ints up to the
    tx.circom size, by their C restatement above it (held equal at the tx.circom size here and in tests/test_oracle_c.py)."""
    from oracle import cbind
    nc, npub = synth.SHAPES[shape]
    t0 = time.time()
    r1, w = synth.generate(nc, npub, seed=11)
    pk_bin, vk = keygen.synth_setup(gp.ctx, r1, TOXIC)
    key = gp.load_key(pk_bin)
    m = gp.key_info(key)["domainSize"]
    wbin = np.frombuffer(synth.witness_bytes(w), dtype=np.uint8)
    rng = random.Random(5)
    r, s = rng.randrange(R), rng.randrange(R)
    got, stats = gp.prove(key, wbin, r, s)
    again, _ = gp.prove(key, wbin, r, s)
    assert got == again
    print("\n%s: m=2^%d nVars=%d prove %.2f ms (setup+gen %.1f s) stats=%s" % (
        shape, m.bit_length() - 1, r1.nVars, stats["total_ms"], time.time() - t0, stats))
    proof = g.proof_from_bytes(got)
    mats = r1.with_input_rows()
    sums = cbind.exponent_sums(mats, r1.pool, npub, wbin, TOXIC[0], m)
    if shape in ("withdraw", "tx"):
        assert sums == g.exponent_sums_flat(mats, r1.pool, npub, w, TOXIC, m)
    assert g.exponent_check_flat(mats, r1.pool, npub, w, TOXIC, m, proof, r, s, sums=sums)
    pub = w[1:npub + 1]
    bad = list(pub)
    bad[-1] = (bad[-1] + 1) % R
    if shape != "tx_2p22":                       # the Python pairing verifier's vk_x loop is per public input
        assert g.verify(vk, proof, pub)
        assert not g.verify(vk, proof, bad)
    vkey = gp.load_vkey(vk["bin"])               # the library's verifier (GPU vk_x MSM + host pairing product)
    assert gp.verify(vkey, got, pub)
    assert not gp.verify(vkey, got, bad)
    zero, _ = gp.prove(key, wbin, 0, 0)          # snarkjs debug mode
    assert g.exponent_check_flat(mats, r1.pool, npub, w, TOXIC, m, g.proof_from_bytes(zero), 0, 0, sums=sums)
    gp.L.zkr_pkey_free(key)
    gp._keys.remove(key)


def test_prove_dev_flags_and_prove_check(gp):
    """zkr_prove_dev is asynchronous and cannot return ZKR_E_WITNESS_RANGE: the flags stay set until zkr_prove_check reads
    them, and a later zkr_prove starts from clean flags (ADVICE r1: a stale flag failed the next valid proof once)."""
    import ctypes as C
    L = gp.L
    r1, w = synth.generate(60, 2, seed=13)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    n = r1.nVars
    good = np.frombuffer(bf.binarify_witness(w), dtype=np.uint8)
    w_bad = list(w)
    w_bad[4] = R                                         # out of range
    bad = np.frombuffer(bf.binarify_witness(w_bad), dtype=np.uint8)
    d_w, d_p = C.c_void_p(), C.c_void_p()
    _lib.check(L.zkr_dev_malloc(gp.ctx, 32 * n, C.byref(d_w)))
    _lib.check(L.zkr_dev_malloc(gp.ctx, 256, C.byref(d_p)))
    rb = np.frombuffer(int(5).to_bytes(32, "little"), dtype=np.uint8)
    sb = np.frombuffer(int(6).to_bytes(32, "little"), dtype=np.uint8)
    want = g.proof_to_bytes(g.gen_proof(pk, w, 5, 6)[0])
    # valid input: OK and the right bytes
    _lib.check(L.zkr_dev_upload(gp.ctx, d_w, _lib.buf_ptr(good), good.size))
    _lib.check(L.zkr_prove_dev(gp.ctx, key, d_w, n, _lib.buf_ptr(rb), _lib.buf_ptr(sb), d_p))
    assert L.zkr_prove_check(gp.ctx, key) == 0
    out = np.zeros(256, dtype=np.uint8)
    _lib.check(L.zkr_dev_download(gp.ctx, _lib.buf_ptr(out), d_p, 256))
    assert out.tobytes() == want
    # invalid input: the call itself succeeds, the check reports it once, then the flags are clean again
    _lib.check(L.zkr_dev_upload(gp.ctx, d_w, _lib.buf_ptr(bad), bad.size))
    assert L.zkr_prove_dev(gp.ctx, key, d_w, n, _lib.buf_ptr(rb), _lib.buf_ptr(sb), d_p) == 0
    assert L.zkr_prove_check(gp.ctx, key) == -3
    assert L.zkr_prove_check(gp.ctx, key) == 0
    # an unchecked bad zkr_prove_dev must not fail the next blocking proof
    assert L.zkr_prove_dev(gp.ctx, key, d_w, n, _lib.buf_ptr(rb), _lib.buf_ptr(sb), d_p) == 0
    got, _ = gp.prove(key, good, 5, 6)
    assert got == want
    _lib.check(L.zkr_dev_free(gp.ctx, d_w))
    _lib.check(L.zkr_dev_free(gp.ctx, d_p))


def test_default_blinding_is_random_and_valid(gp):
    """prove() without r, s (NULL at the C-ABI) draws CSPRNG scalars like websnark: two proofs of the same statement differ
    and both verify; explicit zeros give the deterministic snarkjs debug proof."""
    import ctypes as C
    r1, w = synth.generate(80, 3, seed=14)
    pk, vk, _ = g.setup(r1.to_dicts(), TOXIC)
    key = gp.load_key(bf.binarify_proving_key(pk))
    wb = bf.binarify_witness(w)
    a, _ = gp.prove(key, wb)
    b, _ = gp.prove(key, wb)
    assert a != b
    pub = w[1:4]
    assert g.verify(vk, g.proof_from_bytes(a), pub) and g.verify(vk, g.proof_from_bytes(b), pub)
    z1, _ = gp.prove(key, wb, 0, 0)
    z2, _ = gp.prove(key, wb, 0, 0)
    assert z1 == z2 == g.proof_to_bytes(g.gen_proof(pk, w, 0, 0)[0])
    # NULL straight at the C-ABI
    out1, out2 = np.zeros(256, dtype=np.uint8), np.zeros(256, dtype=np.uint8)
    warr = np.frombuffer(wb, dtype=np.uint8)
    for o in (out1, out2):
        _lib.check(gp.L.zkr_prove(gp.ctx, key, _lib.buf_ptr(warr), r1.nVars, None, None, _lib.buf_ptr(o), None))
    assert out1.tobytes() != out2.tobytes()
    assert g.verify(vk, g.proof_from_bytes(out1.tobytes()), pub)


def test_genproof_key_cache(gp):
    """genProof caches the resident key per (prover, key object / key bytes): repeated calls do not load the key again,
    a different circuit is never served a stale key (ADVICE r1)."""
    r1, w = synth.generate(40, 2, seed=15)
    r2, w2 = synth.generate(40, 2, seed=16)
    pk1, vk1, _ = g.setup(r1.to_dicts(), TOXIC)
    pk2, vk2, _ = g.setup(r2.to_dicts(), TOXIC)
    j1, j2 = bf.pk_to_json(pk1), bf.pk_to_json(pk2)
    n0 = len(gp._keys)
    o1 = prover.genProof(j1, w, 3, 4, prover=gp)
    o1b = prover.genProof(j1, w, 3, 4, prover=gp)
    assert len(gp._keys) == n0 + 1 and o1 == o1b
    o2 = prover.genProof(j2, w2, 3, 4, prover=gp)
    assert len(gp._keys) == n0 + 2
    assert bf.proof_from_json(o1["proof"]) == g.gen_proof(pk1, w, 3, 4)[0]
    assert bf.proof_from_json(o2["proof"]) == g.gen_proof(pk2, w2, 3, 4)[0]
    b1 = bf.binarify_proving_key(pk1)
    prover.genProof(b1, w, 3, 4, prover=gp)
    prover.genProof(bytes(b1), w, 3, 4, prover=gp)
    assert len(gp._keys) == n0 + 3                       # the binary form is cached by content, not reloaded per call


def test_bench_dump_outputs(gp, tmp_path):
    """bench.py --dump-outputs on the withdraw shape: the GPU arm's last timed proof equals what the C port of the
    reference algorithm (--impl reference) writes for the same seeded workload, and it verifies."""
    import json
    import os
    import subprocess
    import sys
    import bench
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    env = dict(os.environ, TMPDIR=str(tmp_path))          # the reference arm's key file: fresh, outside the tree
    arms = (("ours", ["--no-cpu", "--no-gpu-witness", "--no-two-in-flight"]), ("reference", ["--ref-threads", "2"]))
    for impl, extra in arms:
        p = subprocess.run([sys.executable, path, "--impl", impl, "--shape", "withdraw", "--steps", "2", "--warmup", "1",
                            "--dump-outputs", str(tmp_path / impl)] + extra, capture_output=True, text=True, env=env,
                           timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
    got, want = (np.load(tmp_path / impl / "proof.npy") for impl, _ in arms)
    assert got.dtype == np.float64 and got.shape == (8, 32)
    assert np.array_equal(got, want)
    r1, w = synth.generate(*synth.SHAPES["withdraw"], seed=11)
    _, vk = keygen.synth_setup(gp.ctx, r1, bench.TOXIC)
    assert gp.verify(gp.load_vkey(vk["bin"]), got.astype(np.uint8).tobytes(), w[1:r1.nPublic + 1])
