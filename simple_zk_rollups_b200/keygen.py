"""Proving / verifying keys for rollup-shaped R1CS, made on the GPU.

Stands where the reference runs `snarkjs setup --protocol groth` (prover/package.json:34,37).  synth_setup takes the
toxic waste as an explicit input, so its keys are TEST / BENCHMARK keys.  setup_from_powers builds the key from a
public powers-of-tau ceremony and contribute() re-randomises delta (phase 2); verify_contribution() checks a
contribution.  Such a key is sound once at least one contributor erased their delta'.  Output is the websnark
binary proving key -- byte-identical to binarifyProvingKey(snarkjs pk JSON) for the same
(R1CS, toxic waste) -- plus the verifying key as Python ints (and as the binary block zkr_vkey_load_bin takes, vk["bin"]).
The powers themselves come from phase 1 here too: powers_new() is the empty ceremony, powers_contribute() adds one
contribution, powers_verify_contribution() checks one, and powers_verify() checks the powers before setup_from_powers.
"""
import ctypes as C
import struct

import numpy as np

from . import _lib
from .binarify import Q, R

_RINV_Q = pow(1 << 256, -1, Q)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _pols_section(ptr, row, cid, pool_mont_u32, n):
    """writeTransformedPolynomial x n (binarify.ts:104-113,170-177), vectorised."""
    nnz = int(row.size)
    words = np.zeros(n + 9 * nnz, dtype=np.uint32)
    ptr64 = ptr.astype(np.int64)
    words[np.arange(n, dtype=np.int64) + 9 * ptr64[:-1]] = (ptr64[1:] - ptr64[:-1]).astype(np.uint32)
    if nnz:
        sig = np.repeat(np.arange(n, dtype=np.int64), (ptr64[1:] - ptr64[:-1]))
        base = sig + 1 + 9 * np.arange(nnz, dtype=np.int64)
        words[base] = row
        words[(base + 1)[:, None] + np.arange(8)] = pool_mont_u32[cid]
    return words.view(np.uint8)


def _g1(buf):
    x = int.from_bytes(buf[:32], "little") * _RINV_Q % Q
    y = int.from_bytes(buf[32:64], "little") * _RINV_Q % Q
    return None if x == 0 else (x, y)


def _g2(buf):
    v = [int.from_bytes(buf[32 * i:32 * i + 32], "little") * _RINV_Q % Q for i in range(4)]
    return None if v[0] == 0 and v[1] == 0 else ((v[0], v[1]), (v[2], v[3]))


def _r1cs_desc(r1cs):
    """(zkr_r1cs_csc, csc dict, arrays to keep alive) for r1cs with the input-consistency rows in polsA."""
    n, l = r1cs.nVars, r1cs.nPublic
    bits, m = r1cs.domain()
    csc = r1cs.csc(with_inputs=True)
    keep = []
    desc = _lib.R1csCsc()
    desc.n_vars, desc.n_public, desc.n_constraints, desc.domain_size = n, l, r1cs.nConstraints, m
    desc.n_pool = len(r1cs.pool)
    for k in "abc":
        ptr, row, cid = (_u32(x) for x in csc[k.upper()])
        keep += [ptr, row, cid]
        setattr(desc, "ptr_" + k, ptr.ctypes.data)
        setattr(desc, "row_" + k, row.ctypes.data)
        setattr(desc, "cid_" + k, cid.ctypes.data)
    pool = np.frombuffer(b"".join(int(c).to_bytes(32, "little") for c in r1cs.pool), dtype=np.uint8).copy()
    keep.append(pool)
    desc.pool = pool.ctypes.data
    return desc, csc, keep


def _outputs(n, l, m):
    """out_a, out_b1, out_b2, out_c, out_h, out_vk host buffers (zkr.h zkr_synth_setup)."""
    return (np.empty(64 * n, dtype=np.uint8), np.empty(64 * n, dtype=np.uint8), np.empty(128 * n, dtype=np.uint8),
            np.empty(64 * (n - l - 1), dtype=np.uint8), np.empty(64 * m, dtype=np.uint8),
            np.empty(192 + 384 + 64 * (l + 1), dtype=np.uint8))


def vk_dict(vkb, n_public):
    """The verifying key as Python ints from its binary block (alfa1|beta1|delta1|beta2|gamma2|delta2|IC, Fq-M)."""
    vkb = bytes(vkb)
    return dict(protocol="groth", nPublic=n_public, vk_alfa_1=_g1(vkb[0:64]), vk_beta_2=_g2(vkb[192:320]),
                vk_gamma_2=_g2(vkb[320:448]), vk_delta_2=_g2(vkb[448:576]),
                IC=[_g1(vkb[576 + 64 * i:640 + 64 * i]) for i in range(n_public + 1)],
                bin=vkb)                 # the block zkr_vkey_load_bin takes


def _assemble(r1cs, csc, out_a, out_b1, out_b2, out_c, out_h, out_vk):
    """websnark binary proving key (binarify.ts:152-202) around the point sections, and the vk dict."""
    n, l = r1cs.nVars, r1cs.nPublic
    bits, m = r1cs.domain()
    pool_mont = np.frombuffer(b"".join(((int(c) << 256) % R).to_bytes(32, "little") for c in r1cs.pool),
                              dtype=np.uint32).reshape(-1, 8)
    secA = _pols_section(*[_u32(x) for x in csc["A"]], pool_mont, n)
    secB = _pols_section(*[_u32(x) for x in csc["B"]], pool_mont, n)
    vkb = out_vk.tobytes()
    fixed = vkb[0:192] + vkb[192:320] + vkb[448:576]          # alfa1 beta1 delta1 | beta2 | delta2
    ptrs, off = [], 40 + len(fixed)
    for sec in (secA, secB, out_a, out_b1, out_b2, out_c, out_h):
        ptrs.append(off)
        off += sec.size
    if off >= 1 << 32:
        raise ValueError("websnark binary key offsets are u32 (binarify.ts:155-161): key too large")
    head = struct.pack("<10I", n, l, m, *ptrs)
    pk_bin = np.concatenate([np.frombuffer(head + fixed, dtype=np.uint8), secA, secB, out_a, out_b1, out_b2,
                             out_c, out_h])
    assert pk_bin.size == off
    return pk_bin, vk_dict(vkb, l)


def synth_setup(ctx, r1cs, toxic):
    """r1cs: simple_zk_rollups_b200.synth.R1CS; toxic = (tau, alpha, beta, gamma, delta) ints.
    -> (pk_bin: np.ndarray[uint8], vk: dict of int points)."""
    L = _lib.lib()
    desc, csc, keep = _r1cs_desc(r1cs)
    outs = _outputs(r1cs.nVars, r1cs.nPublic, r1cs.domain()[1])
    tox = np.frombuffer(b"".join(int(t % R).to_bytes(32, "little") for t in toxic), dtype=np.uint8).copy()
    _lib.check(L.zkr_synth_setup(ctx, C.byref(desc), _lib.buf_ptr(tox), *[_lib.buf_ptr(x) for x in outs]))
    return _assemble(r1cs, csc, *outs)


_POWER_SECTIONS = (("tau_g1", 64), ("tau_g2", 128), ("alpha_tau_g1", 64), ("beta_tau_g1", 64))


def _powers_desc(powers, keep):
    """zkr_powers for a powers dict; the buffers it points to are appended to keep."""
    pw = _lib.Powers()
    for name, size in _POWER_SECTIONS + (("beta_g2", 128),):
        buf = np.frombuffer(bytes(powers[name]), dtype=np.uint8)
        if buf.size % size:
            raise ValueError("%s: %d bytes is not a whole number of %d-byte points" % (name, buf.size, size))
        keep.append(buf)
        setattr(pw, name, buf.ctypes.data if buf.size else None)
        if name != "beta_g2":
            setattr(pw, "n_" + name, min(buf.size // size, 0xFFFFFFFF))
        elif buf.size != 128:
            raise ValueError("beta_g2 must be one 128-byte G2 point")
    return pw


def setup_from_powers(ctx, r1cs, powers):
    """Circuit key from phase-1 powers of tau (zkr_setup_from_powers; zkr.h has the math and the security statement).
    powers: dict of byte buffers (bytes / uint8 arrays) of affine Fq-M points in the key encoding: "tau_g1"
    (>= 2m - 1 points, 2m for H_(m-1)), "tau_g2", "alpha_tau_g1", "beta_tau_g1" (>= m each) and "beta_g2" (one point).
    -> (pk_bin, vk) as synth_setup, for gamma = delta = 1: NOT deployable before one contribute()."""
    L = _lib.lib()
    desc, csc, keep = _r1cs_desc(r1cs)
    pw = _powers_desc(powers, keep)
    outs = _outputs(r1cs.nVars, r1cs.nPublic, r1cs.domain()[1])
    _lib.check(L.zkr_setup_from_powers(ctx, C.byref(desc), C.byref(pw), *[_lib.buf_ptr(x) for x in outs]))
    return _assemble(r1cs, csc, *outs)


def _vk_bin(vk):
    return np.frombuffer(bytes(vk["bin"] if isinstance(vk, dict) else vk), dtype=np.uint8)


def contribute(ctx, pk_bin, vk, delta=None):
    """One phase-2 contribution (zkr_setup_contribute): delta1, delta2 times delta', C and H times 1/delta'.
    delta: int in [1, r) (tests, reproducible keys) or None = drawn from the OS CSPRNG and never seen by Python.
    -> (new pk_bin, new vk dict, 96-byte record R | z proving knowledge of delta')."""
    L = _lib.lib()
    pk = np.ascontiguousarray(pk_bin, dtype=np.uint8)
    vkb = _vk_bin(vk)
    out_pk = np.empty_like(pk)
    out_vk = np.empty_like(vkb)
    rec = np.empty(_lib.CONTRIB_RECORD_BYTES, dtype=np.uint8)
    d = None if delta is None else int(delta).to_bytes(32, "little")
    _lib.check(L.zkr_setup_contribute(ctx, _lib.buf_ptr(pk), pk.size, _lib.buf_ptr(vkb), vkb.size, _lib.buf_ptr(d),
                                      _lib.buf_ptr(out_pk), _lib.buf_ptr(out_vk), _lib.buf_ptr(rec)))
    n_public = struct.unpack_from("<I", pk[:8].tobytes(), 4)[0]
    return out_pk, vk_dict(out_vk, n_public), rec.tobytes()


def verify_contribution(ctx, old_pk, old_vk, new_pk, new_vk, record):
    """True iff (new_pk, new_vk) is (old_pk, old_vk) after the contribution `record` proves (zkr.h lists the checks)."""
    L = _lib.lib()
    po = np.ascontiguousarray(old_pk, dtype=np.uint8)
    pn = np.ascontiguousarray(new_pk, dtype=np.uint8)
    vo, vn = _vk_bin(old_vk), _vk_bin(new_vk)
    rec = bytes(record)
    if pn.size != po.size or vn.size != vo.size or len(rec) != _lib.CONTRIB_RECORD_BYTES:
        raise ValueError("old and new keys differ in size, or the record is not %d bytes" % _lib.CONTRIB_RECORD_BYTES)
    valid = C.c_int(0)
    _lib.check(L.zkr_setup_verify_contribution(ctx, _lib.buf_ptr(po), _lib.buf_ptr(vo), _lib.buf_ptr(pn),
                                               _lib.buf_ptr(vn), po.size, vo.size, _lib.buf_ptr(rec),
                                               C.byref(valid)))
    return bool(valid.value)


# ------------------------------------------------------------------------------------------------ phase 1
def _gen_points(ctx, group, n):
    one = (1).to_bytes(32, "little")
    out = np.empty(64 if group == 1 else 128, dtype=np.uint8)
    _lib.check(_lib.lib().zkr_synth_points(ctx, group, _lib.buf_ptr(one), 1, _lib.buf_ptr(out)))
    return out.tobytes() * n


def powers_new(ctx, m, n_tau_g1=None):
    """The empty ceremony (tau = alpha = beta = 1): every point a generator; tau_g1 has n_tau_g1 points (default 2m),
    tau_g2, alpha_tau_g1 and beta_tau_g1 m each.  A powers dict as setup_from_powers takes."""
    n_tau_g1 = 2 * m if n_tau_g1 is None else n_tau_g1
    return {"tau_g1": _gen_points(ctx, 1, n_tau_g1), "tau_g2": _gen_points(ctx, 2, m),
            "alpha_tau_g1": _gen_points(ctx, 1, m), "beta_tau_g1": _gen_points(ctx, 1, m),
            "beta_g2": _gen_points(ctx, 2, 1)}


def powers_contribute(ctx, powers, tau=None, alpha=None, beta=None):
    """One phase-1 contribution (zkr_powers_contribute): the powers of (tau tau', alpha alpha', beta beta').
    tau, alpha, beta: ints in [1, r) (tests, reproducible transcripts), or all None = drawn from the OS CSPRNG and never
    seen by Python.  -> (new powers dict, 288-byte record: Schnorr proofs of knowledge of tau', alpha', beta')."""
    given = [x is not None for x in (tau, alpha, beta)]
    if any(given) and not all(given):
        raise ValueError("give all three secrets or none")
    keep = []
    pw = _powers_desc(powers, keep)
    out = {name: np.empty(len(bytes(powers[name])), dtype=np.uint8) for name, _ in _POWER_SECTIONS + (("beta_g2", 128),)}
    rec = np.empty(_lib.POWERS_RECORD_BYTES, dtype=np.uint8)
    sec = None if tau is None else b"".join(int(x).to_bytes(32, "little") for x in (tau, alpha, beta))
    _lib.check(_lib.lib().zkr_powers_contribute(ctx, C.byref(pw), _lib.buf_ptr(sec), *[
        _lib.buf_ptr(out[name]) for name in ("tau_g1", "tau_g2", "alpha_tau_g1", "beta_tau_g1", "beta_g2")],
        _lib.buf_ptr(rec)))
    return {name: buf.tobytes() for name, buf in out.items()}, rec.tobytes()


def _verdict(valid):
    return (True, "") if valid.value else (False, _lib.lib().zkr_last_error().decode())


def powers_verify(ctx, powers):
    """(ok, reason): ok iff the powers are well formed (zkr_powers_verify lists the checks); reason names the first
    failed check."""
    keep = []
    pw = _powers_desc(powers, keep)
    valid = C.c_int(0)
    _lib.check(_lib.lib().zkr_powers_verify(ctx, C.byref(pw), C.byref(valid)))
    return _verdict(valid)


def powers_verify_contribution(ctx, old, new, record):
    """(ok, reason): ok iff `new` is `old` after the contribution `record` proves, and `new` is well formed."""
    rec = bytes(record)
    if len(rec) != _lib.POWERS_RECORD_BYTES:
        raise ValueError("the record is not %d bytes" % _lib.POWERS_RECORD_BYTES)
    keep = []
    po, pn = _powers_desc(old, keep), _powers_desc(new, keep)
    valid = C.c_int(0)
    _lib.check(_lib.lib().zkr_powers_verify_contribution(ctx, C.byref(po), C.byref(pn), _lib.buf_ptr(rec),
                                                         C.byref(valid)))
    return _verdict(valid)
