"""ctypes binding of oracle/c/libzkr_oracle.so (the C restatement of the reference prove path).
TEST INFRASTRUCTURE ONLY -- see oracle/c/zkr_oracle.c."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "c", "libzkr_oracle.so")
_lib = None


def build(force=False):
    src = [os.path.join(HERE, "c", f) for f in ("zkr_oracle.c", "curve_tmpl.h", "Makefile")]
    if force or not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in src):
        subprocess.run(["make", "-C", os.path.join(HERE, "c"), "-B", "libzkr_oracle.so"], check=True,
                       capture_output=True)
    return SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            build()
        L = C.CDLL(SO)
        L.oracle_ntt.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.oracle_h_from_evals.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.oracle_msm.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int]
        L.oracle_prove.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.oracle_field_mul.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.oracle_ap_points.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.oracle_exponent_sums.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p]
        L.oracle_horner.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.oracle_g1_add.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.oracle_g1_mul.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _p(b):
    if b is None:
        return None
    if isinstance(b, bytes):
        return C.cast(C.c_char_p(b), C.c_void_p)
    return C.c_void_p(b.ctypes.data)          # numpy


def prove(pk_bin, witness_bin, r=0, s=0, mode=1, threads=None, want_h=False):
    """-> 256-byte proof (and the m x 32 B standard-form h vector if want_h)."""
    import numpy as np
    threads = threads or os.cpu_count() or 1
    pk = np.frombuffer(pk_bin, dtype=np.uint8) if isinstance(pk_bin, (bytes, bytearray)) else pk_bin
    w = np.frombuffer(witness_bin, dtype=np.uint8) if isinstance(witness_bin, (bytes, bytearray)) else witness_bin
    out = np.zeros(256, dtype=np.uint8)
    m = int(np.frombuffer(pk[8:12].tobytes(), dtype=np.uint32)[0])
    h = np.zeros(32 * m, dtype=np.uint8) if want_h else None
    rb = np.frombuffer(int(r).to_bytes(32, "little"), dtype=np.uint8)
    sb = np.frombuffer(int(s).to_bytes(32, "little"), dtype=np.uint8)
    rc = lib().oracle_prove(_p(pk), pk.size, _p(w), w.size // 32, _p(rb), _p(sb), _p(out), mode, threads, _p(h))
    if rc != 0:
        raise RuntimeError("oracle_prove failed: %d" % rc)
    return (out.tobytes(), h) if want_h else out.tobytes()


def msm(group, points_mont, scalars, mode=1, threads=None):
    import numpy as np
    threads = threads or os.cpu_count() or 1
    n = scalars.size // 32
    out = np.zeros(64 if group == 1 else 128, dtype=np.uint8)
    lib().oracle_msm(group, _p(points_mont), _p(scalars), n, _p(out), mode, threads)
    return out.tobytes()


def ntt(data, bits, inverse=False, coset=False, mode=1, threads=None):
    threads = threads or os.cpu_count() or 1
    lib().oracle_ntt(_p(data), bits, int(inverse), int(coset), mode, threads)
    return data


def h_from_evals(at, bt, bits, mode=1, threads=None):
    """h of calcH (websnark's 2m-point method) from A_T, B_T: numpy uint8, 2^bits x 32 B standard form each -> the same."""
    import numpy as np
    threads = threads or os.cpu_count() or 1
    at, bt = np.ascontiguousarray(at, dtype=np.uint8), np.ascontiguousarray(bt, dtype=np.uint8)
    assert at.size == bt.size == 32 << bits
    out = np.zeros(32 << bits, dtype=np.uint8)
    lib().oracle_h_from_evals(_p(at), _p(bt), bits, _p(out), mode, threads)
    return out


def ap_points(group, base_mont, step_mont, n):
    """P_i = base + i * step, i < n -> n x 64 / 128 B affine Fq-M (numpy uint8).  base / step: affine Fq-M bytes."""
    import numpy as np
    out = np.zeros(n * (64 if group == 1 else 128), dtype=np.uint8)
    lib().oracle_ap_points(group, _p(bytes(base_mont)), _p(bytes(step_mont)), n, _p(out))
    return out


def horner(coeffs, x):
    """sum_j coeffs[j] x^j mod r; coeffs: numpy uint8 (n x 32 B standard form), x: int -> int."""
    import numpy as np
    out = np.zeros(32, dtype=np.uint8)
    xb = np.frombuffer(int(x).to_bytes(32, "little"), dtype=np.uint8)
    lib().oracle_horner(_p(coeffs), coeffs.size // 32, _p(xb), _p(out))
    return int.from_bytes(out.tobytes(), "little")


def g1_add(p_mont, q_mont):
    import numpy as np
    out = np.zeros(64, dtype=np.uint8)
    lib().oracle_g1_add(_p(bytes(p_mont)), _p(bytes(q_mont)), _p(out))
    return out.tobytes()


def g1_mul(p_mont, k):
    import numpy as np
    out = np.zeros(64, dtype=np.uint8)
    lib().oracle_g1_mul(_p(bytes(p_mont)), _p(int(k).to_bytes(32, "little")), _p(out))
    return out.tobytes()


def exponent_sums(mats, pool, n_public, witness_bin, tau, m):
    """C restatement of the sparse pass of oracle.groth16.exponent_check_flat: -> (tot, priv) dicts of ints keyed
    "A" / "B" / "C" (pass them as sums= to exponent_check_flat).  witness_bin: n x 32 B standard form."""
    import numpy as np
    w = np.frombuffer(witness_bin, dtype=np.uint8) if isinstance(witness_bin, (bytes, bytearray)) else witness_bin
    pb = np.frombuffer(b"".join(int(c).to_bytes(32, "little") for c in pool), dtype=np.uint8)
    tb = np.frombuffer(int(tau).to_bytes(32, "little"), dtype=np.uint8)
    tot, priv = {}, {}
    for name, (sig, row, cid) in mats.items():
        sig, row, cid = (np.ascontiguousarray(a, dtype=np.uint32) for a in (sig, row, cid))
        t, p = np.zeros(32, dtype=np.uint8), np.zeros(32, dtype=np.uint8)
        lib().oracle_exponent_sums(m.bit_length() - 1, _p(tb), _p(w), _p(pb), len(pool), _p(sig), _p(row), _p(cid),
                                   sig.size, n_public, _p(t), _p(p))
        tot[name] = int.from_bytes(t.tobytes(), "little")
        priv[name] = int.from_bytes(p.tobytes(), "little")
    return tot, priv
