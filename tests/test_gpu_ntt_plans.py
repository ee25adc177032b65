"""GPU NTT and H pipeline on every pass plan, whole vectors against host references, byte for byte.

Which kernel geometry a transform runs (csrc/ntt.cu, plan_passes / ntt_run_ex), with the default knobs:
  2^1 - 2^2    k_ntt_tiny
  2^3 - 2^11   one pass
  2^12 - 2^22  two passes, tiles narrowed to one column (c = 0) to make 1024 CTAs, full twiddle table for pass 0
  2^23 - 2^24  three passes (8/8/7, 8/8/8) with multi-column tiles (c = 11 - k) in passes 0 and 1; the middle pass's
               full twiddle table is built with tw_shift > 0
  2^25 up      three passes, two-level (tlo / thi) twiddle lookup
ZKR_NTT_MIN_BLOCKS (0: full-width tiles), ZKR_NTT_TWFULL_MAXLOG (0: two-level lookup at every size), ZKR_NTT_SPLIT
(explicit pass widths) and ZKR_H_UNFUSED (round-1 H pipeline) are read once per process: those arms run in child
processes.  2^26 and 2^27 are left to bench.py's sharded rows: their host reference takes minutes.

References: the Python oracle (recursive radix-2) up to 2^14; above, the oracle's C NTT (iterative, threaded; held equal
to the Python one by test_oracle_c.py).  The H pipeline is held to the oracle's C calcH, websnark's 2m-point method rather
than the L/U split the GPU uses, and under the split arms to the Python oracle's calc_h_lu."""
import ctypes as C
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import cbind
from oracle import groth16 as g
from oracle.bn254 import R
from simple_zk_rollups_b200 import _lib
from helpers import MONT, bitrev_rows, full_range, pack, unpack

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FWD, INV, CFWD, CINV = 0, 1, 2, 3
BR_OUT, BR_IN = 0x10, 0x20
ALL_MODES = (FWD, INV, CFWD, CINV)
PY_MAX = 14                  # the Python oracle is the reference up to 2^14
CACHE_MAX = 23               # inputs and references reused by the knob arms are kept for the module up to 2^23
ON_DEVICE = (2, 9, 16, 23, 25)   # one size per plan class also runs every mode through on_device = 1
# one mode per kernel variant: DIF forward, DIF inverse (natural in), DIT inverse, DIT forward (bit-reversed in)
ARM_MODES = (FWD, CINV, INV | BR_IN, CFWD | BR_IN)


def runs(log_n):
    """(mode | order) list of the default-plan test: every mode in every order to 2^22; the orders the prover chains at
    2^23 and 2^24; at 2^25 forward and coset inverse (1 GB per vector)."""
    if log_n <= 22:
        return [m | o for m in ALL_MODES for o in (0, BR_OUT, BR_IN)]
    if log_n <= 24:
        return list(ALL_MODES) + [m | o for m in (FWD, INV) for o in (BR_OUT, BR_IN)]
    return [FWD, CINV]


def host_ntt(x, log_n, base):
    """natural-order transform of x (flat uint8, 2^log_n x 32 B standard form) by the host reference"""
    if log_n <= PY_MAX:
        v, sh = unpack(x), g.root_of_unity(log_n + 1)
        return pack({FWD: lambda: g.ntt(v), INV: lambda: g.ntt(v, inverse=True), CFWD: lambda: g.coset_ntt(v, sh),
                     CINV: lambda: g.coset_intt(v, sh)}[base]())
    return cbind.ntt(x.copy(), log_n, base in (INV, CINV), base in (CFWD, CINV))


def _frozen(a):
    a.setflags(write=False)
    return a


@functools.lru_cache(maxsize=None)
def _uniform_cached(log_n):
    return _frozen(full_range(1 << log_n, log_n))


@functools.lru_cache(maxsize=None)
def _want_cached(log_n, base):
    return _frozen(host_ntt(_uniform_cached(log_n), log_n, base))


def uniform(log_n):
    return _uniform_cached(log_n) if log_n <= CACHE_MAX else full_range(1 << log_n, log_n)


def want_uniform(log_n, base):
    return _want_cached(log_n, base) if log_n <= CACHE_MAX else host_ntt(uniform(log_n), log_n, base)


def h_inputs(log_m):
    """full-range A_T, B_T of the H tests at 2^log_m"""
    return full_range(1 << log_m, 1000 + log_m), full_range(1 << log_m, 2000 + log_m)


@functools.lru_cache(maxsize=None)
def want_h(log_m):
    return _frozen(cbind.h_from_evals(*h_inputs(log_m), log_m))


@functools.lru_cache(maxsize=None)
def want_h_lu(log_m):
    at, bt = (unpack(v) for v in h_inputs(log_m))
    m = 1 << log_m
    pk = dict(domainSize=m, polsA=[{i: at[i] for i in range(m)}], polsB=[{i: bt[i] for i in range(m)}])
    return _frozen(pack(g.calc_h_lu(pk, [1])))


@pytest.fixture(scope="module", autouse=True)
def _drop_caches():
    yield
    for f in (_uniform_cached, _want_cached, want_h, want_h_lu):
        f.cache_clear()


def expect_equal(got, want, what):
    if not np.array_equal(got, want):
        bad = np.flatnonzero((got.reshape(-1, 32) != want.reshape(-1, 32)).any(axis=1))
        pytest.fail("%s: %d of %d elements differ, first at %s" % (what, bad.size, want.size // 32, bad[:8].tolist()))


def arrange(x, want_nat, log_n, mode):
    """-> (input, expected output) of one run: BITREV_IN takes its input in bit-reversed order, BITREV_OUT leaves its
    output so"""
    return (bitrev_rows(x, log_n) if mode & BR_IN else x,
            bitrev_rows(want_nat, log_n) if mode & BR_OUT else want_nat)


class DevBuf:
    def __init__(self, zctx, nbytes):
        self.zctx, self.p = zctx, C.c_void_p()
        _lib.check(_lib.lib().zkr_dev_malloc(zctx, nbytes, C.byref(self.p)))

    def upload(self, host):
        _lib.check(_lib.lib().zkr_dev_upload(self.zctx, self.p, _lib.buf_ptr(host), host.size))

    def download(self, nbytes):
        out = np.zeros(nbytes, dtype=np.uint8)
        _lib.check(_lib.lib().zkr_dev_download(self.zctx, _lib.buf_ptr(out), self.p, nbytes))
        return out

    def free(self):
        _lib.check(_lib.lib().zkr_dev_free(self.zctx, self.p))


def gpu_ntt(zctx, x, log_n, mode, on_device=False):
    if not on_device:
        buf = x.copy()
        _lib.check(_lib.lib().zkr_ntt(zctx, _lib.buf_ptr(buf), log_n, mode, 0))
        return buf
    d = DevBuf(zctx, x.size)
    try:
        d.upload(x)
        _lib.check(_lib.lib().zkr_ntt(zctx, d.p, log_n, mode, 1))
        return d.download(x.size)
    finally:
        d.free()


def gpu_h(zctx, at, bt, log_m, bitrev):
    nb = at.size
    bufs = [DevBuf(zctx, nb) for _ in range(3)]
    try:
        bufs[0].upload(at)
        bufs[1].upload(bt)
        _lib.check(_lib.lib().zkr_h_from_evals_dev(zctx, bufs[0].p, bufs[1].p, log_m, bufs[2].p, bitrev))
        return bufs[2].download(nb)
    finally:
        for b in bufs:
            b.free()


# ------------------------------------------------------------------------------------------------ default plans
@pytest.mark.parametrize("log_n", range(1, 26))
def test_ntt_default_plan(zctx, log_n):
    """Full-range input (r - 1, 0, 1 first, r - 1 last) in every mode and order of runs(log_n), whole output against the
    host reference; at one size per plan class (ON_DEVICE) every run also goes through on_device = 1."""
    x = uniform(log_n)
    for base in ALL_MODES:
        modes = [m for m in runs(log_n) if m & 0xF == base]
        if not modes:
            continue
        want = want_uniform(log_n, base)
        for mode in modes:
            inp, exp = arrange(x, want, log_n, mode)
            expect_equal(gpu_ntt(zctx, inp, log_n, mode), exp, "2^%d mode %#x" % (log_n, mode))
            if log_n in ON_DEVICE:
                expect_equal(gpu_ntt(zctx, inp, log_n, mode, on_device=True), exp,
                             "2^%d mode %#x on device" % (log_n, mode))


def check_geometric(got, a, b, what):
    """got == [a b^k]_k, the whole vector: got[0] == a and got[k + 1] == got[k] b, the products taken by the oracle's C
    Montgomery multiplication (standard-form got[k] times b R gives got[k] b)."""
    n = got.size // 32
    assert unpack(got[:32]) == [a], what + ": index 0"
    step = 1 << 20
    bm = np.tile(pack([b * MONT % R]), min(step, n))
    for lo in range(0, n - 1, step):
        cnt = min(step, n - 1 - lo)
        cur = np.ascontiguousarray(got[32 * lo:32 * (lo + cnt)])
        nxt = np.zeros(32 * cnt, dtype=np.uint8)
        cbind.lib().oracle_field_mul(1, cur.ctypes.data, bm.ctypes.data, nxt.ctypes.data, cnt)
        expect_equal(got[32 * (lo + 1):32 * (lo + 1 + cnt)], nxt, "%s: indices %d.." % (what, lo + 1))


@pytest.mark.parametrize("log_n", range(1, 26))
def test_ntt_closed_form(zctx, log_n):
    """Inputs whose transforms are known in closed form, forward and inverse (every order to 2^22, natural above):
    a constant c -> (c n, 0, ..., 0) / (c, 0, ..., 0), the same with c = r - 1, and e_(n-1) -> X[k] = w^-k / w^k / n.
    Both the constant and e_(n-1) are their own bit reversal, so BITREV_IN takes the same input."""
    n = 1 << log_n
    orders = (0, BR_OUT, BR_IN) if log_n <= 22 else (0,)
    for val in (0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF % R, R - 1):
        x = np.tile(pack([val]), n)
        for base, x0 in ((FWD, val * n % R), (INV, val)):
            exp = np.zeros(32 * n, dtype=np.uint8)
            exp[:32] = pack([x0])
            for o in orders:
                expect_equal(gpu_ntt(zctx, x, log_n, base | o), exp, "2^%d constant %#x mode %#x" % (log_n, val, base | o))
        del x, exp
    x = np.zeros(32 * n, dtype=np.uint8)
    x[-32] = 1
    w = g.root_of_unity(log_n)
    for base, a, b in ((FWD, 1, pow(w, -1, R)), (INV, pow(n, -1, R), w)):
        for o in orders:
            got = gpu_ntt(zctx, x, log_n, base | o)
            check_geometric(bitrev_rows(got, log_n) if o == BR_OUT else got, a, b, "2^%d e_(n-1) mode %#x" % (log_n, base | o))


# ------------------------------------------------------------------------------------------------ H pipeline, every size
@pytest.mark.parametrize("log_m", range(1, 24))
def test_h_pipeline_every_size(zctx, log_m):
    """zkr_h_from_evals_dev on full-range A_T, B_T against the oracle's C calcH (websnark's method), in both output
    orders; A_T = B_T = r - 1 (A B = 1, so h = 0) too."""
    at, bt = h_inputs(log_m)
    want = want_h(log_m)
    for bitrev in (0, 1):
        expect_equal(gpu_h(zctx, at, bt, log_m, bitrev), bitrev_rows(want, log_m) if bitrev else want,
                     "h 2^%d bitrev_out %d" % (log_m, bitrev))
    rm1 = np.tile(pack([R - 1]), 1 << log_m)
    for bitrev in (0, 1):
        assert not gpu_h(zctx, rm1, rm1, log_m, bitrev).any(), "h 2^%d of r - 1, bitrev_out %d" % (log_m, bitrev)


# ------------------------------------------------------------------------------------------------ knob arms (child processes)
_CHILD = r"""
import ctypes as C, json, os, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from simple_zk_rollups_b200 import _lib
d = sys.argv[2]
L = _lib.lib()
ctx = C.c_void_p()
_lib.check(L.zkr_ctx_create(0, C.byref(ctx)))
ld = lambda name: np.fromfile(os.path.join(d, name), dtype=np.uint8)
for job in json.load(open(os.path.join(d, "jobs.json"))):
    if job["kind"] == "ntt":
        buf = ld(job["x"])
        _lib.check(L.zkr_ntt(ctx, _lib.buf_ptr(buf), job["log"], job["mode"], 0))
    else:
        a, b = ld(job["a"]), ld(job["b"])
        p = [C.c_void_p() for _ in range(3)]
        for q in p:
            _lib.check(L.zkr_dev_malloc(ctx, a.size, C.byref(q)))
        _lib.check(L.zkr_dev_upload(ctx, p[0], _lib.buf_ptr(a), a.size))
        _lib.check(L.zkr_dev_upload(ctx, p[1], _lib.buf_ptr(b), b.size))
        _lib.check(L.zkr_h_from_evals_dev(ctx, p[0], p[1], job["log"], p[2], job["bitrev"]))
        buf = np.zeros(a.size, dtype=np.uint8)
        _lib.check(L.zkr_dev_download(ctx, _lib.buf_ptr(buf), p[2], a.size))
        for q in p:
            _lib.check(L.zkr_dev_free(ctx, q))
    buf.tofile(os.path.join(d, job["out"]))
L.zkr_ctx_destroy(ctx)
"""


class Arm:
    """Transforms and H pipelines run by one child process under knob settings; inputs and outputs go through files in
    tmp_path, expectations stay here."""

    def __init__(self, tmp_path):
        self.d, self.jobs, self.expect, self.nfiles = tmp_path, [], [], 0

    def _file(self, arr):
        name = "in%d.bin" % self.nfiles
        self.nfiles += 1
        arr.tofile(self.d / name)
        return name

    def ntt(self, log_n, mode, x, want_nat):
        inp, exp = arrange(x, want_nat, log_n, mode)
        self.jobs.append(dict(kind="ntt", log=log_n, mode=mode, x=self._file(inp), out="out%d.bin" % len(self.jobs)))
        self.expect.append((exp, "2^%d mode %#x" % (log_n, mode)))

    def h(self, log_m, bitrev, want):
        at, bt = h_inputs(log_m)
        self.jobs.append(dict(kind="h", log=log_m, bitrev=bitrev, a=self._file(at), b=self._file(bt),
                              out="out%d.bin" % len(self.jobs)))
        self.expect.append((bitrev_rows(want, log_m) if bitrev else want, "h 2^%d bitrev_out %d" % (log_m, bitrev)))

    def run(self, **knobs):
        (self.d / "jobs.json").write_text(json.dumps(self.jobs))
        env = {k: v for k, v in os.environ.items() if not k.startswith(("ZKR_NTT_", "ZKR_H_"))}
        env.update(knobs)
        p = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(self.d)], capture_output=True, text=True, env=env,
                           timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        for job, (exp, what) in zip(self.jobs, self.expect):
            expect_equal(np.fromfile(self.d / job["out"], dtype=np.uint8), exp, "%s under %s" % (what, knobs))


def test_ntt_full_width_tiles(tmp_path):
    """ZKR_NTT_MIN_BLOCKS=0: tiles keep their full width, so the first of two passes takes c = 11 - k adjacent columns
    (2^12: c = 5 ... 2^20: c = 1) in both kernel directions; the fused H pipeline on the same tiles."""
    arm = Arm(tmp_path)
    for log_n in range(12, 21):
        for mode in ARM_MODES:
            arm.ntt(log_n, mode, uniform(log_n), want_uniform(log_n, mode & 0xF))
    for log_m in (12, 16, 20):
        for bitrev in (0, 1):
            arm.h(log_m, bitrev, want_h(log_m))
    arm.run(ZKR_NTT_MIN_BLOCKS="0")


def test_ntt_two_level_twiddles(tmp_path):
    """ZKR_NTT_TWFULL_MAXLOG=0: the inter-pass twiddles come from the two-level lookup at two-pass sizes and at 2^23
    (three passes, multi-column tiles, tw_shift > 0 in the middle pass); the H pipeline at 2^12 and 2^23 on it."""
    arm = Arm(tmp_path)
    for log_n in (12, 17, 22, 23):
        for mode in ARM_MODES:
            arm.ntt(log_n, mode, uniform(log_n), want_uniform(log_n, mode & 0xF))
    for log_m in (12, 23):
        arm.h(log_m, 1, want_h(log_m))
    arm.run(ZKR_NTT_TWFULL_MAXLOG="0")


@pytest.mark.parametrize("split", ["3,3,3", "3,3,3,3", "5,4,3", "11,3", "3,11"])
def test_ntt_split_plans(tmp_path, split):
    """ZKR_NTT_SPLIT (with ZKR_NTT_MIN_BLOCKS=0, so the tiles take c > 0 columns): three- and four-pass plans, and an
    11-bit pass beside a 3-bit one in both orders, at sizes the Python oracle handles; every mode in every order, and
    the H pipeline (three and four passes, fused) against calc_h_lu."""
    log_n = sum(int(k) for k in split.split(","))
    arm = Arm(tmp_path)
    x = uniform(log_n)
    for mode in runs(log_n):
        arm.ntt(log_n, mode, x, want_uniform(log_n, mode & 0xF))
    for bitrev in (0, 1):
        arm.h(log_n, bitrev, want_h_lu(log_n))
    arm.run(ZKR_NTT_SPLIT=split, ZKR_NTT_MIN_BLOCKS="0")


def test_h_unfused(tmp_path):
    """ZKR_H_UNFUSED=1: the round-1 H pipeline (element-wise sweeps between plain transforms) with bit-reversed output,
    at one, two and three passes."""
    arm = Arm(tmp_path)
    for log_m in (3, 11, 12, 17, 23):
        arm.h(log_m, 1, want_h(log_m))
    arm.run(ZKR_H_UNFUSED="1")
