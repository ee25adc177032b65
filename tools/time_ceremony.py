"""Device time of the ceremony setup (csrc/ceremony.cu): setup_from_powers at the tx.circom shape (m = 2^17) and the
2^20 rollup shape, contribute and verify_contribution at 2^20.  Synthetic powers for known (tau, alpha, beta), so each
timed key is also checked byte for byte against synth_setup(tau, alpha, beta, 1, delta).  Each call is blocking; CUDA
events are recorded on the current stream before and after it.  The card's name and power limit are read in the same
run.  Writes one JSON file.   python tools/time_ceremony.py --out profiles/r03_setup_ceremony.json [--reps 2]"""
import argparse
import json
import os
import random
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from simple_zk_rollups_b200 import _lib, keygen, prover, synth  # noqa: E402

R = synth.R


def synthetic_powers(ctx, m, tau, alpha, beta):
    def pts(group, scalars):
        sc = np.frombuffer(b"".join(s.to_bytes(32, "little") for s in scalars), dtype=np.uint8)
        out = np.empty(len(scalars) * (64 if group == 1 else 128), dtype=np.uint8)
        _lib.check(_lib.lib().zkr_synth_points(ctx, group, _lib.buf_ptr(sc), len(scalars), _lib.buf_ptr(out)))
        return out.tobytes()

    tp = [1]
    for _ in range(2 * m - 1):
        tp.append(tp[-1] * tau % R)
    return {"tau_g1": pts(1, tp), "tau_g2": pts(2, tp[:m]), "alpha_tau_g1": pts(1, [alpha * t % R for t in tp[:m]]),
            "beta_tau_g1": pts(1, [beta * t % R for t in tp[:m]]), "beta_g2": pts(2, [beta])}


def timed(fn, reps):
    """[ms per call] from CUDA events around each blocking call, and the last result."""
    out, res = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = fn()
        b.record()
        b.synchronize()
        out.append(round(a.elapsed_time(b), 1))
    return out, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    torch.cuda.init()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    rec = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi, "reps": a.reps, "rows": []}
    gp = prover.Groth16Prover(0)
    rng = random.Random(2026)
    tau, alpha, beta, delta = (rng.randrange(1, R) for _ in range(4))
    try:
        for shape in ("tx", "tx_2p20"):
            r1, _ = synth.generate(*synth.SHAPES[shape])
            bits, m = r1.domain()
            pw = synthetic_powers(gp.ctx, m, tau, alpha, beta)
            keygen.setup_from_powers(gp.ctx, r1, pw)                   # warm-up: module load, twiddle tables
            ms, (pk, vk) = timed(lambda: keygen.setup_from_powers(gp.ctx, r1, pw), a.reps)
            ref = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, 1))
            same = bytes(pk) == bytes(ref[0]) and bytes(vk["bin"]) == bytes(ref[1]["bin"])
            row = {"shape": shape, "m": m, "n_vars": r1.nVars, "nnz": r1.nnz(), "setup_from_powers_ms": ms,
                   "identical_to_synth_setup": same}
            if shape == "tx_2p20":
                ms_c, (pk1, vk1, recd) = timed(lambda: keygen.contribute(gp.ctx, pk, vk, delta), a.reps)
                ms_v, ok = timed(lambda: keygen.verify_contribution(gp.ctx, pk, vk, pk1, vk1, recd), a.reps)
                ref = keygen.synth_setup(gp.ctx, r1, (tau, alpha, beta, 1, delta))
                row.update(contribute_ms=ms_c, verify_contribution_ms=ms_v, verified=ok,
                           contribution_identical_to_synth_setup=bytes(pk1) == bytes(ref[0]) and
                           bytes(vk1["bin"]) == bytes(ref[1]["bin"]))
            rec["rows"].append(row)
            print(json.dumps(row), flush=True)
    finally:
        gp.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "power": smi}))


if __name__ == "__main__":
    main()
