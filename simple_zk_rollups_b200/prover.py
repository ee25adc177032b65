"""Python host mirror of the reference's proof-generator API, backed by libzkr (CUDA, sm_100a).

Reference surface kept (operator/src/snarks/common.ts:10-53, tx.ts:6-10, withdraw.ts:6-10):
    createProofGenerator(provingKey, verifyingKey, circuitName) -> async (circuitInputs) ->
        {proof, solidityProof: {a, b, c, inputs}}
and the snarkjs-shaped call the north star names:
    genProof(provingKey, witness) -> {proof: {pi_a, pi_b, pi_c, protocol}, publicSignals}
What changes underneath: common.ts:23 (buildBn128), :28 (binarifyProvingKey per proof) and :29
(groth16GenProof) become one resident key + zkr_prove.  Witness generation (common.ts:12-21) and the
self-verification (common.ts:30-38) stay host-side callables exactly as they stay TypeScript in the
reference; circom cannot run here, so the witness calculator is an injected callable.
No CPU fallback: every prove goes through the CUDA library or raises.
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from .binarify import R as SNARK_FIELD_SIZE
from .binarify import binarifyProvingKey, binarifyWitness, proof_from_bytes, proof_to_bytes


class Groth16Prover:
    """One libzkr context (one GPU) with proving keys resident in HBM."""

    def __init__(self, device=0):
        self.L = _lib.lib()
        self.ctx = C.c_void_p()
        _lib.check(self.L.zkr_ctx_create(device, C.byref(self.ctx)))
        self.device = device
        self._keys = []
        self._vkeys = []
        self._manys = []

    def close(self):
        for h in list(self._manys):                   # workspaces share their key's tables: freed before the keys
            h.close()
        for k in self._keys:
            self.L.zkr_pkey_free(k)
        self._keys = []
        for k in self._vkeys:
            self.L.zkr_vkey_free(k)
        self._vkeys = []
        if self.ctx:
            self.L.zkr_ctx_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def load_key(self, pk_bin):
        """pk_bin: bytes / numpy uint8 in the binarifyProvingKey layout.  Parsed + uploaded once."""
        arr = np.frombuffer(pk_bin, dtype=np.uint8) if isinstance(pk_bin, (bytes, bytearray)) else pk_bin
        h = C.c_void_p()
        _lib.check(self.L.zkr_pkey_load_bin(self.ctx, _lib.buf_ptr(arr), arr.size, C.byref(h)))
        self._keys.append(h)
        return h

    def load_key_json(self, text):
        """text: the snarkjs proving_key.json TEXT (str / bytes).  Native parse + binarify + upload, once."""
        data = text.encode() if isinstance(text, str) else bytes(text)
        h = C.c_void_p()
        _lib.check(self.L.zkr_pkey_load_json(self.ctx, data, len(data), C.byref(h)))
        self._keys.append(h)
        return h

    def load_vkey(self, verifyingKey):
        """verifyingKey: snarkjs verification_key.json as dict / JSON text, or the binary vk block of
        keygen.synth_setup (vk["bin"]).  IC tables become resident on this GPU (zkr_vkey_load_*)."""
        import json
        h = C.c_void_p()
        if isinstance(verifyingKey, dict):
            verifyingKey = json.dumps(verifyingKey)
        if isinstance(verifyingKey, str):
            data = verifyingKey.encode()
            _lib.check(self.L.zkr_vkey_load_json(self.ctx, data, len(data), C.byref(h)))
        else:
            arr = np.frombuffer(verifyingKey, dtype=np.uint8) if isinstance(verifyingKey, (bytes, bytearray)) else verifyingKey
            _lib.check(self.L.zkr_vkey_load_bin(self.ctx, _lib.buf_ptr(arr), arr.size, C.byref(h)))
        self._vkeys.append(h)
        return h

    def verify(self, vkey, proof, publicSignals):
        """groth.isValid(vk, proof, publicSignals) (common.ts:30-34) as the on-chain predicate
        (TxVerifier.sol:258-276).  proof: 256-byte buffer or the {pi_a, pi_b, pi_c} object."""
        if isinstance(proof, dict):
            proof = proof_to_bytes(proof)
        pb = np.frombuffer(bytes(proof), dtype=np.uint8)
        pub = np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in publicSignals), dtype=np.uint8)
        ok = C.c_int()
        _lib.check(self.L.zkr_verify(self.ctx, vkey, _lib.buf_ptr(pb), _lib.buf_ptr(pub) if pub.size else None,
                                     len(publicSignals), C.byref(ok)))
        return bool(ok.value)

    def load_key_sharded(self, pk_bin, rank, world):
        """Keep only `rank`'s point range of the five base sets (one proof split over `world` GPUs)."""
        arr = np.frombuffer(pk_bin, dtype=np.uint8) if isinstance(pk_bin, (bytes, bytearray)) else pk_bin
        h = C.c_void_p()
        _lib.check(self.L.zkr_pkey_load_bin_sharded(self.ctx, _lib.buf_ptr(arr), arr.size, rank, world, C.byref(h)))
        self._keys.append(h)
        return h

    def prove_sharded(self, comm, key, witness_bin, r, s):
        """comm: sharding.Comm of this rank (all ranks call with the same witness, r, s) -> (proof, stats);
        every rank returns the same 256 bytes as prove() on one GPU.  r, s are required: the ranks must agree on them,
        so the caller draws them once (secrets.randbelow(r)) and hands the same pair to every rank."""
        w = np.frombuffer(witness_bin, dtype=np.uint8) if isinstance(witness_bin, (bytes, bytearray)) else witness_bin
        out = np.zeros(_lib.PROOF_BYTES, dtype=np.uint8)
        st = _lib.Stats()
        rb = np.frombuffer(int(r).to_bytes(32, "little"), dtype=np.uint8)
        sb = np.frombuffer(int(s).to_bytes(32, "little"), dtype=np.uint8)
        _lib.check(self.L.zkr_prove_sharded(comm.h, key, _lib.buf_ptr(w), w.size // 32, _lib.buf_ptr(rb),
                                            _lib.buf_ptr(sb), _lib.buf_ptr(out), C.byref(st)))
        return out.tobytes(), st.as_dict()

    def key_info(self, key):
        a, b, c, d = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint64()
        _lib.check(self.L.zkr_pkey_info(key, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return dict(nVars=a.value, nPublic=b.value, domainSize=c.value, device_bytes=d.value)

    def prove(self, key, witness_bin, r=None, s=None):
        """witness_bin: binarifyWitness output.  r, s: blinding scalars (ints < r).  None (the default) draws a fresh
        CSPRNG scalar, as websnark's groth16GenProof does internally: proofs are zero-knowledge unless the caller
        asks otherwise.  Pass explicit values for parity tests; (0, 0) is the snarkjs debug mode (deterministic,
        NOT zero-knowledge).  -> (256-byte proof, stats dict)."""
        r = _random_scalar() if r is None else r
        s = _random_scalar() if s is None else s
        w = np.frombuffer(witness_bin, dtype=np.uint8) if isinstance(witness_bin, (bytes, bytearray)) else witness_bin
        out = np.zeros(_lib.PROOF_BYTES, dtype=np.uint8)
        st = _lib.Stats()
        rb = np.frombuffer(int(r).to_bytes(32, "little"), dtype=np.uint8)
        sb = np.frombuffer(int(s).to_bytes(32, "little"), dtype=np.uint8)
        _lib.check(self.L.zkr_prove(self.ctx, key, _lib.buf_ptr(w), w.size // 32, _lib.buf_ptr(rb),
                                    _lib.buf_ptr(sb), _lib.buf_ptr(out), C.byref(st)))
        return out.tobytes(), st.as_dict()

    def kernel_launches(self):
        return int(self.L.zkr_ctx_kernel_launches(self.ctx))

    def create_many(self, key, max_proofs):
        """Work buffers for proving up to max_proofs witnesses of `key` in one pass (zkr_many_create).  The key's
        tables are shared; close the handle before the key is freed."""
        h = C.c_void_p()
        _lib.check(self.L.zkr_many_create(self.ctx, key, int(max_proofs), C.byref(h)))
        m = ManyHandle(self, h)
        self._manys.append(m)
        return m

    def prove_many(self, handle, witness_bins, rs=None):
        """zkr_prove_many: every witness of the list proved in one pass through every stage.  witness_bins:
        binarifyWitness outputs of one key; rs: optional list of (r, s) ints, None draws a fresh CSPRNG pair per proof.
        -> list of 256-byte proofs, proof j byte-identical to prove(key, witness_bins[j], *rs[j])."""
        n = len(witness_bins)
        ws = [np.frombuffer(w, dtype=np.uint8) if isinstance(w, (bytes, bytearray)) else np.asarray(w, dtype=np.uint8)
              for w in witness_bins]
        if n == 0:
            return []
        if any(w.size != ws[0].size for w in ws):
            raise ValueError("all witnesses of a batch must have the same length")
        flat = np.ascontiguousarray(np.concatenate(ws))
        rsb = None
        if rs is not None:
            if len(rs) != n:
                raise ValueError("rs must give one (r, s) pair per witness")
            rsb = np.frombuffer(b"".join(int(r).to_bytes(32, "little") + int(s).to_bytes(32, "little") for r, s in rs),
                                dtype=np.uint8)
        out = np.zeros(n * _lib.PROOF_BYTES, dtype=np.uint8)
        _lib.check(self.L.zkr_prove_many(self.ctx, handle.h, _lib.buf_ptr(flat), ws[0].size // 32, n, _lib.buf_ptr(rsb),
                                         _lib.buf_ptr(out)))
        return [out[i * _lib.PROOF_BYTES:(i + 1) * _lib.PROOF_BYTES].tobytes() for i in range(n)]

    def msm_many(self, bases, scalars, n, n_vectors, group=1):
        """zkr_msm_many: n_vectors MSMs over one base set (a zkr_bases handle of this context).  scalars: n_vectors x n
        x 32 bytes, std form.  -> list of affine std-form results (64 bytes for G1, 128 for G2), one per vector."""
        sc = np.frombuffer(scalars, dtype=np.uint8) if isinstance(scalars, (bytes, bytearray)) else np.ascontiguousarray(scalars)
        ob = 64 if group == 1 else 128
        out = np.zeros(n_vectors * ob, dtype=np.uint8)
        _lib.check(self.L.zkr_msm_many(self.ctx, bases, _lib.buf_ptr(sc), n, n_vectors, 0, _lib.buf_ptr(out)))
        return [out[i * ob:(i + 1) * ob].tobytes() for i in range(n_vectors)]


class ManyHandle:
    """A zkr_many workspace (Groth16Prover.create_many); close() frees it."""

    def __init__(self, prover, h):
        self.prover, self.h = prover, h

    def info(self):
        k, b = C.c_int(), C.c_uint64()
        _lib.check(self.prover.L.zkr_many_info(self.h, C.byref(k), C.byref(b)))
        return dict(max_proofs=k.value, device_bytes=b.value)

    def close(self):
        if self.h:
            self.prover.L.zkr_many_free(self.h)
            self.h = C.c_void_p()
            self.prover._manys.remove(self)


def prove_batch(provers, keys, witness_bins, rs=None):
    """zkr_prove_batch: n independent proofs over len(provers) contexts (one per GPU; keys[i] is the same circuit's
    key loaded on provers[i]), round-robin, one proof in flight per GPU -- the shape of many genTxVerifierProof calls
    (operator/src/snarks/tx.ts:6-10) drained by an operator batch loop.  witness_bins: list of binarifyWitness
    outputs; rs: optional list of (r, s) ints; None draws a fresh CSPRNG pair per proof (pass [(0, 0)] * n for the
    snarkjs debug mode).  -> list of 256-byte proofs, in input order."""
    L = provers[0].L
    n = len(witness_bins)
    if n == 0:
        return []
    ws = [np.frombuffer(w, dtype=np.uint8) if isinstance(w, (bytes, bytearray)) else w for w in witness_bins]
    n_signals = ws[0].size // 32
    if any(w.size != ws[0].size for w in ws):
        raise ValueError("all witnesses of a batch must have the same length")
    ctxs = (C.c_void_p * len(provers))(*[p.ctx for p in provers])
    pks = (C.c_void_p * len(provers))(*keys)
    wptrs = (C.c_void_p * n)(*[w.ctypes.data for w in ws])
    if rs is None:
        rs = [(_random_scalar(), _random_scalar()) for _ in range(n)]
    rsb = None
    if rs is not None:
        rsb = np.frombuffer(b"".join(int(r).to_bytes(32, "little") + int(s).to_bytes(32, "little") for r, s in rs),
                            dtype=np.uint8)
    out = np.zeros(n * _lib.PROOF_BYTES, dtype=np.uint8)
    _lib.check(L.zkr_prove_batch(ctxs, pks, len(provers), wptrs, n_signals, n, _lib.buf_ptr(rsb), _lib.buf_ptr(out)))
    return [out[i * _lib.PROOF_BYTES:(i + 1) * _lib.PROOF_BYTES].tobytes() for i in range(n)]


_default = None


def default_prover():
    global _default
    if _default is None:
        _default = Groth16Prover(0)
    return _default


def _random_scalar():
    import secrets
    return secrets.randbelow(SNARK_FIELD_SIZE)


class _KeyCache:
    """Resident keys of genProof, per (prover, key object).  The entry keeps a reference to the key object it was made
    from, so its id() cannot be recycled for another circuit while the entry lives; byte / array keys are looked up by
    a content hash.  Bounded: the least recently used key is freed on the device (zkr_pkey_free) when a new one would
    exceed `limit` resident keys."""

    def __init__(self, limit=4):
        self.limit, self.entries = limit, {}

    def get(self, p, provingKey):
        import hashlib
        if isinstance(provingKey, dict):
            ck = (id(p), "obj", id(provingKey))
        else:
            buf = provingKey if isinstance(provingKey, (bytes, bytearray)) else np.ascontiguousarray(provingKey).tobytes()
            ck = (id(p), "bin", hashlib.blake2b(buf, digest_size=16).digest(), len(buf))
        e = self.entries.pop(ck, None)
        if e is None or e[0] not in p._keys:             # absent, or freed behind our back (prover.close())
            binkey = binarifyProvingKey(provingKey) if isinstance(provingKey, dict) else provingKey
            key = p.load_key(binkey)
            e = (key, p.key_info(key)["nPublic"], provingKey if isinstance(provingKey, dict) else None, p)
            while len(self.entries) >= self.limit:
                old_key, _, _, old_p = self.entries.pop(next(iter(self.entries)))
                if old_key in old_p._keys:
                    old_p.L.zkr_pkey_free(old_key)
                    old_p._keys.remove(old_key)
        self.entries[ck] = e                             # re-inserted last: most recently used
        return e[0], e[1]


_key_cache = _KeyCache()


def genProof(provingKey, witness, r=None, s=None, prover=None):
    """snarkjs groth.genProof shape: -> {"proof": {pi_a, pi_b, pi_c, protocol}, "publicSignals": [...]}.
    provingKey: snarkjs pk JSON (dict) or an already-binarified key (bytes / uint8 array); the resident key is cached
    per (prover, key) -- callers that prove in a loop should still load the key once (Groth16Prover.load_key) and call
    prove() with the handle.  r, s default to CSPRNG draws like websnark; pass 0, 0 for the snarkjs debug mode."""
    p = prover or default_prover()
    key, n_public = _key_cache.get(p, provingKey)
    buf, _ = p.prove(key, binarifyWitness(witness), r, s)
    return {"proof": proof_from_bytes(buf), "publicSignals": [str(int(x)) for x in witness[1:n_public + 1]]}


def _load_any_key(p, provingKey):
    """snarkjs pk JSON as dict, as JSON text or as a path to proving_key.json (the reference `require`s the file,
    operator/src/snarks/tx.ts:3), or an already binarified key (bytes / uint8 array)."""
    if isinstance(provingKey, dict):
        return p.load_key(binarifyProvingKey(provingKey))
    if isinstance(provingKey, str):
        return p.load_key_json(open(provingKey).read() if os.path.exists(provingKey) else provingKey)
    return p.load_key(provingKey)


def createProofGenerator(provingKey, verifyingKey, circuitName, calculateWitness, isValid=None, prover=None):
    """Mirror of operator/src/snarks/common.ts:10-53.

    calculateWitness(circuitName, circuitInputs) -> (witness: list[int], nPubInputs_plus_nOutputs: int)
        stands for circom compile + snarkjs Circuit.calculateWitness (common.ts:12-21), which stay
        on the host in the reference as well.
    isValid(verifyingKey, proof, publicSignals) -> bool stands for snarkjs groth.isValid
        (common.ts:30-34); an invalid proof raises "Invalid proof generated" (common.ts:36-38).  Default:
        the library's own verifier (zkr_verify, the TxVerifier.sol:258-276 predicate) on verifyingKey;
        pass verifyingKey=None to skip the self-check.
    The returned callable is synchronous; the reference's is async only because websnark is."""
    p = prover or default_prover()
    key = _load_any_key(p, provingKey)
    if isinstance(verifyingKey, str) and os.path.exists(verifyingKey):
        verifyingKey = open(verifyingKey).read()
    if isValid is None and verifyingKey is not None:
        vkey = p.load_vkey(verifyingKey)             # once per circuit; IC tables resident on the GPU

        def isValid(_vk, proof, publicSignals):      # noqa: F811  (zkr_verify: GPU vk_x + host pairing product)
            return p.verify(vkey, proof, publicSignals)

    def generate(circuitInputs, r=None, s=None):
        witness, n_pub = calculateWitness(circuitName, circuitInputs)
        publicSignals = witness[1:n_pub + 1]
        buf, _ = p.prove(key, binarifyWitness(witness), r, s)
        proof = proof_from_bytes(buf)
        if isValid is not None and not isValid(verifyingKey, proof, publicSignals):
            raise RuntimeError("Invalid proof generated")
        return {
            "proof": proof,
            "solidityProof": {                       # common.ts:42-50
                "a": proof["pi_a"][:2],
                "b": [list(reversed(x)) for x in proof["pi_b"]][:2],
                "c": proof["pi_c"][:2],
                "inputs": [str(int(x) % SNARK_FIELD_SIZE) for x in publicSignals],
            },
        }

    return generate


def bindCircuit(buildDir, name, calculateWitness, prover=None):
    """Mirror of the reference's thin binders (operator/src/snarks/tx.ts:1-10, withdraw.ts:1-10):
        genTxVerifierProof       = bindCircuit(build, "tx", calc)        # txProvingKey.json / txVerifyingKey.json
        genWithdrawVerifierProof = bindCircuit(build, "withdraw", calc)  # withdrawProvingKey.json / ...
    buildDir is the reference's prover/build directory; the key files are parsed natively, once."""
    return createProofGenerator(os.path.join(buildDir, "%sProvingKey.json" % name),
                                os.path.join(buildDir, "%sVerifyingKey.json" % name),
                                "%s.circom" % name, calculateWitness, prover=prover)
