"""ctypes binding of libzkr.so (the C-ABI in include/zkr.h).  No torch, no oracle, no CPU fallback:
if the library is missing or no B200 is visible, calls raise ZkrError."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# ZKR_LIB: load a variant build instead (simple_zk_rollups_b200/build.py, A/B of compile-time choices on one GPU box)
LIB_PATH = os.environ.get("ZKR_LIB") or os.path.join(HERE, "libzkr.so")

PROOF_BYTES = 256
CONTRIB_RECORD_BYTES = 96
POWERS_RECORD_BYTES = 288


class ZkrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libzkr error %d: %s" % (code, msg))
        self.code = code


class Stats(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "total_ms", "h2d_ms", "lc_ms", "ntt_ms", "msm_a_ms", "msm_b1_ms", "msm_b2_ms",
        "msm_c_ms", "msm_h_ms", "assemble_ms")] + [("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class R1csCsc(C.Structure):
    _fields_ = [("n_vars", C.c_uint32), ("n_public", C.c_uint32), ("n_constraints", C.c_uint32),
                ("domain_size", C.c_uint32), ("n_pool", C.c_uint32)] + \
               [(n, C.c_void_p) for n in ("ptr_a", "row_a", "cid_a", "ptr_b", "row_b", "cid_b",
                                          "ptr_c", "row_c", "cid_c", "pool")]


class Powers(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("n_tau_g1", "n_tau_g2", "n_alpha_tau_g1", "n_beta_tau_g1")] + \
               [(n, C.c_void_p) for n in ("tau_g1", "tau_g2", "alpha_tau_g1", "beta_tau_g1", "beta_g2")]


_SIGS = {
    "zkr_strerror": (C.c_char_p, [C.c_int]),
    "zkr_last_error": (C.c_char_p, []),
    "zkr_version": (C.c_char_p, []),
    "zkr_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "zkr_ctx_destroy": (None, [C.c_void_p]),
    "zkr_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "zkr_ctx_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "zkr_ctx_set_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "zkr_ctx_set_serial": (C.c_int, [C.c_void_p, C.c_int]),
    "zkr_ctx_profile_read": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int),
                                       C.POINTER(C.c_double)]),
    "zkr_dev_malloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_dev_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zkr_dev_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zkr_pkey_load_bin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_pkey_free": (None, [C.c_void_p]),
    "zkr_pkey_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "zkr_pkey_json_to_bin": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "zkr_witness_json_to_bin": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "zkr_buf_free": (None, [C.c_void_p]),
    "zkr_pkey_load_json": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_vkey_load_json": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_vkey_load_bin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_vkey_free": (None, [C.c_void_p]),
    "zkr_vkey_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "zkr_verify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "zkr_pairing_check": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "zkr_prove": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                            C.c_void_p, C.POINTER(Stats)]),
    "zkr_prove_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "zkr_prove_check": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_fill_geometric": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int,
                                     C.c_int, C.c_int]),
    "zkr_wprog_build": (C.c_int, [C.c_void_p, C.POINTER(R1csCsc), C.POINTER(C.c_void_p)]),
    "zkr_wprog_free": (None, [C.c_void_p]),
    "zkr_wprog_info": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_uint32)] * 4),
    "zkr_wprog_given": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_witness_solve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zkr_prove_batch": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                  C.POINTER(C.c_void_p), C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]),
    "zkr_many_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "zkr_many_free": (None, [C.c_void_p]),
    "zkr_many_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "zkr_prove_many": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]),
    "zkr_msm_many": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]),
    "zkr_bases_load": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "zkr_bases_free": (None, [C.c_void_p]),
    "zkr_bases_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.c_uint64)]),
    "zkr_msm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "zkr_msm_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "zkr_ntt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "zkr_h_from_evals_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "zkr_comm_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]),
    "zkr_comm_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zkr_comm_connect_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "zkr_comm_barrier": (C.c_int, [C.c_void_p]),
    "zkr_comm_check": (C.c_int, [C.c_void_p]),
    "zkr_comm_buffer": (C.c_void_p, [C.c_void_p, C.c_int]),
    "zkr_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "zkr_comm_destroy": (None, [C.c_void_p]),
    "zkr_msm_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "zkr_pkey_load_bin_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "zkr_shard_ranges": (C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]),
    "zkr_prove_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.POINTER(Stats)]),
    "zkr_ntt_sharded_rows_log": (C.c_int, [C.c_int, C.c_int]),
    "zkr_ntt_sharded": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "zkr_synth_setup": (C.c_int, [C.c_void_p, C.POINTER(R1csCsc), C.c_void_p] + [C.c_void_p] * 6),
    "zkr_setup_from_powers": (C.c_int, [C.c_void_p, C.POINTER(R1csCsc), C.POINTER(Powers)] + [C.c_void_p] * 6),
    "zkr_setup_contribute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "zkr_setup_verify_contribution": (C.c_int, [C.c_void_p] + [C.c_void_p] * 4 + [C.c_size_t, C.c_size_t, C.c_void_p,
                                                                                  C.POINTER(C.c_int)]),
    "zkr_powers_contribute": (C.c_int, [C.c_void_p, C.POINTER(Powers), C.c_void_p] + [C.c_void_p] * 6),
    "zkr_powers_verify": (C.c_int, [C.c_void_p, C.POINTER(Powers), C.POINTER(C.c_int)]),
    "zkr_powers_verify_contribution": (C.c_int, [C.c_void_p, C.POINTER(Powers), C.POINTER(Powers), C.c_void_p,
                                                 C.POINTER(C.c_int)]),
    "zkr_synth_points": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "zkr_test_field_op": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zkr_test_curve_op": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zkr_test_bases_peek": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t]),
    "zkr_microbench": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
}

_lib = None


def exported_names():
    return sorted(_SIGS)


def lib():
    """Load libzkr.so (once).  Raises if it has not been built -- never falls back to anything."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ZkrError(-5, "libzkr.so not built (run `python -m simple_zk_rollups_b200.build`); "
                               "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name, None)    # tests/test_abi.py asserts none is missing
            if f is None:
                continue
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise ZkrError(rc, lib().zkr_last_error().decode() or lib().zkr_strerror(rc).decode())


def buf_ptr(b):
    """void* for bytes / bytearray / numpy array / int (already a pointer) / None."""
    if b is None:
        return None
    if isinstance(b, int):
        return C.c_void_p(b)
    if isinstance(b, bytes):
        return C.cast(C.c_char_p(b), C.c_void_p)
    if isinstance(b, bytearray):
        return C.c_void_p(C.addressof(C.c_char.from_buffer(b)))
    if hasattr(b, "ctypes"):
        return C.c_void_p(b.ctypes.data)
    return C.cast(b, C.c_void_p)
