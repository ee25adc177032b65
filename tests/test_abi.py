"""CPU tests: the C-ABI library loads without a GPU, exports every symbol include/zkr.h declares, fails
loudly (no CPU fallback), and the product never imports the oracle."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from simple_zk_rollups_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "zkr.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(zkr_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    names = _declared()
    assert len(names) >= 25
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert sorted(set(_lib.exported_names())) == names, "ctypes signature table out of sync with zkr.h"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (zkr_[a-z0-9_]+)", out))
    assert set(names) <= exported


def test_version_and_strerror():
    L = _lib.lib()
    assert b"sm_100a" in L.zkr_version()
    assert L.zkr_strerror(0) == b"ok" and b"no CPU fallback" in L.zkr_strerror(-5)


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible here")
    L = _lib.lib()
    h = C.c_void_p()
    rc = L.zkr_ctx_create(0, C.byref(h))
    assert rc == -5 and not h.value
    assert b"no CPU fallback" in L.zkr_last_error()
    from simple_zk_rollups_b200 import prover
    with pytest.raises(_lib.ZkrError):
        prover.Groth16Prover(0)
    assert L.zkr_pkey_load_bin(None, None, 0, C.byref(h)) == -1
    assert L.zkr_ntt(None, None, 3, 0, 0) == -1


def test_product_does_not_touch_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs may use oracle/."""
    pkg = os.path.join(ROOT, "simple_zk_rollups_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".ts", ".cc", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(dirpath, f)
                assert "zkr_oracle" not in txt and "libzkr_oracle" not in txt, os.path.join(dirpath, f)
    code = ("import sys; sys.path.insert(0, %r); import simple_zk_rollups_b200.prover, simple_zk_rollups_b200.keygen, "
            "simple_zk_rollups_b200.synth, simple_zk_rollups_b200.binarify; "
            "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules)" % ROOT)
    subprocess.run([sys.executable, "-c", code], check=True)


def test_napi_addon_source_compiles_and_serialises_ctx_calls():
    """The N-API shim is shipped as source (no node in the image): compile it against a declarations-only node_api.h
    and check that every zkr_* call on the shared context sits under the addon's mutex (zkr.h: calls on one ctx are
    serialised by the caller; ADVICE r1: overlapping `await zkr.prove()` raced on the key's work buffers)."""
    src = os.path.join(ROOT, "simple_zk_rollups_b200", "ts", "zkr_napi.cc")
    p = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Wno-comment", "-Werror",
                        "-I", os.path.join(ROOT, "tests", "csrc", "napi_stub"), "-I", os.path.join(ROOT, "include"), src],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    lines = open(src).read().splitlines()
    for i, ln in enumerate(lines):
        m = re.search(r"\b(zkr_(?!last_error|strerror|ctx\b|pkey\b|vkey\b)\w+)\(", ln)
        if not m or ln.lstrip().startswith("//"):
            continue
        window = "\n".join(lines[max(0, i - 6):i])
        assert "Lock lk(g_mu)" in window, "%s at line %d is not under g_mu" % (m.group(1), i + 1)


def test_bench_contract_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout


def test_bench_dump_proof_layout(tmp_path):
    """bench.py --dump-outputs: the 256 proof bytes as float64 (8 coordinates x 32 bytes), exact and in order."""
    import numpy as np
    import bench
    proof = bytes((7 * i + 3) % 256 for i in range(256))
    bench.dump_proof(str(tmp_path / "out"), "proof", proof)
    a = np.load(tmp_path / "out" / "proof.npy")
    assert a.dtype == np.float64 and a.shape == (8, 32)
    assert a.astype(np.uint8).tobytes() == proof and np.array_equal(a, np.round(a))


def test_sharded_rows_log_python_mirror_matches_library():
    """pure host logic of the sharded NTT plan (no GPU needed): the Python mirror equals the library."""
    import os
    from simple_zk_rollups_b200 import _lib, sharding as sh
    assert "ZKR_NTT_SHARD_K0" not in os.environ
    L = _lib.lib()
    for world in (1, 2, 4, 8):
        for log_n in range(8, 28):
            assert L.zkr_ntt_sharded_rows_log(log_n, world) == sh.rows_log_default(log_n, world), (log_n, world)
