"""Proofs per second of zkr_prove_many (csrc/prover.cu: k witnesses of one key in one pass) against zkr_prove_batch with
one and with two contexts, at the withdraw (2 763 constraints, m = 2^12) and tx (m = 2^17) shapes.

Witnesses are distinct (a few signals of the synthetic witness changed: well formed, circuit-violating, which the prover
must reproduce all the same), in host memory, with fixed distinct (r, s).  Every call is blocking; CUDA events are
recorded on the current stream before and after it, after one warm-up call of the same k.  Every timed proof is checked
byte for byte against zkr_prove on the same inputs.  The card's name and power limit are read in the same run.  The
withdraw key (47.5 MB) fits in the B200's 126 MB L2, and so do the batch buffers of a few proofs (the file's `memory`
records their size), so the withdraw timings are of a largely L2-resident working set.  Writes one JSON file.
    python tools/time_prove_many.py --out profiles/r03_prove_many.json [--reps 3]"""
import argparse
import json
import os
import random
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from simple_zk_rollups_b200 import keygen, prover, synth  # noqa: E402

R = synth.R
TOXIC = (1234567891011, 222222222222223, 3333333333333331, 44444444444447, 5555555555555557)
KS = {"withdraw": (1, 8, 32, 128, 256), "tx": (1, 8, 32, 128)}


def timed(fn, reps):
    """[ms per call] from CUDA events around each blocking call, and the last result (one untimed warm-up first)."""
    fn()
    out, res = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = fn()
        b.record()
        b.synchronize()
        out.append(round(a.elapsed_time(b), 3))
    return out, res


def witnesses(w, k, rng):
    """k distinct binarified witnesses: 4 private signals of w replaced by random values < 2^64 (< r)."""
    base = np.frombuffer(synth.witness_bytes(w), dtype=np.uint8)
    out = []
    for j in range(k):
        x = base.copy()
        for i in rng.sample(range(1, len(w)), 4):
            x[32 * i:32 * i + 32] = np.frombuffer(rng.getrandbits(64).to_bytes(8, "little") + bytes(24), dtype=np.uint8)
        out.append(x)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    torch.cuda.init()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    rec = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi, "reps": a.reps,
           "timing": "CUDA events around each blocking call, after one warm-up call of the same k; host witness buffers",
           "rows": []}
    gp, gp2 = prover.Groth16Prover(0), prover.Groth16Prover(0)
    rng = random.Random(2026)
    try:
        for shape, ks in KS.items():
            nc, npub = synth.SHAPES[shape]
            r1, w = synth.generate(nc, npub, seed=11)
            pk_bin, _ = keygen.synth_setup(gp.ctx, r1, TOXIC)
            key, key2 = gp.load_key(pk_bin), gp2.load_key(pk_bin)
            info = gp.key_info(key)
            h = gp.create_many(key, max(ks))
            many_bytes = h.info()["device_bytes"]
            for k in ks:
                ws = witnesses(w, k, rng)
                rs = [(rng.randrange(R), rng.randrange(R)) for _ in range(k)]
                want = [gp.prove(key, x, r, s)[0] for x, (r, s) in zip(ws, rs)]
                ms_many, got = timed(lambda: gp.prove_many(h, ws, rs), a.reps)
                ms_b1, got_b1 = timed(lambda: prover.prove_batch([gp], [key], ws, rs), a.reps)
                ms_b2, got_b2 = timed(lambda: prover.prove_batch([gp, gp2], [key, key2], ws, rs), a.reps)
                row = {"shape": shape, "n_vars": info["nVars"], "domain_size": info["domainSize"], "k": k,
                       "prove_many_ms": ms_many, "prove_many_proofs_per_s": round(1000 * k / min(ms_many), 1),
                       "prove_batch_1ctx_ms": ms_b1, "prove_batch_1ctx_proofs_per_s": round(1000 * k / min(ms_b1), 1),
                       "prove_batch_2ctx_ms": ms_b2, "prove_batch_2ctx_proofs_per_s": round(1000 * k / min(ms_b2), 1),
                       "identical_to_zkr_prove": got == want and got_b1 == want and got_b2 == want}
                rec["rows"].append(row)
                print(json.dumps(row), flush=True)
                assert row["identical_to_zkr_prove"], row
            rec.setdefault("memory", []).append({
                "shape": shape, "key_device_bytes": info["device_bytes"], "max_proofs": max(ks),
                "many_device_bytes": many_bytes, "many_device_bytes_per_proof": many_bytes // max(ks)})
            h.close()
            for p, kk in ((gp, key), (gp2, key2)):
                p.L.zkr_pkey_free(kk)
                p._keys.remove(kk)
    finally:
        gp2.close()
        gp.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"gpu": rec["gpu"], "power": smi, "memory": rec["memory"]}))


if __name__ == "__main__":
    main()
