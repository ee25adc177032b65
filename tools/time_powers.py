"""Device time of phase 1 (csrc/powers.cu): powers_contribute, powers_verify and powers_verify_contribution at the
tx.circom ceremony (m = 2^17: 2^18 G1 powers, 2^17 of the others) and the 2^20 rollup one.  Synthetic powers for known
(tau, alpha, beta), so every timed contribution is also checked byte for byte against the synthetic powers of
(tau tau', alpha alpha', beta beta').  Each call is blocking; CUDA events are recorded on the current stream before and
after it.  The card's name and power limit are read in the same run.  Writes one JSON file.
    python tools/time_powers.py --out profiles/r03_powers_ceremony.json [--reps 2]"""
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
    old_s = [rng.randrange(1, R) for _ in range(3)]
    new_s = [rng.randrange(1, R) for _ in range(3)]
    try:
        for name, log_m in (("tx", 17), ("tx_2p20", 20)):
            m = 1 << log_m
            old = synthetic_powers(gp.ctx, m, *old_s)
            want = synthetic_powers(gp.ctx, m, *[x * y % R for x, y in zip(old_s, new_s)])
            keygen.powers_contribute(gp.ctx, old, *new_s)                        # warm-up: module load
            ms_c, (new, record) = timed(lambda: keygen.powers_contribute(gp.ctx, old, *new_s), a.reps)
            same = all(bytes(new[k]) == bytes(want[k]) for k in want)
            ms_v, verdict = timed(lambda: keygen.powers_verify(gp.ctx, new), a.reps)
            ms_vc, verdict_c = timed(lambda: keygen.powers_verify_contribution(gp.ctx, old, new, record), a.reps)
            row = {"shape": name, "m": m, "n_tau_g1": 2 * m, "n_tau_g2": m, "n_alpha_tau_g1": m, "n_beta_tau_g1": m,
                   "contribute_ms": ms_c, "verify_ms": ms_v, "verify_contribution_ms": ms_vc,
                   "identical_to_synthetic_powers": same, "verified": verdict[0], "contribution_verified": verdict_c[0]}
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
