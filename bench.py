#!/usr/bin/env python3
"""Benchmark of the Groth16 prove hot path (BASELINE.json metric: "BN254 Groth16 prove ms + proofs/s; ...").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape tx_2p20] [--dump-outputs DIR]

One "step" = one complete proof (witness -> 256-byte proof) of the rollup-shaped circuit named in
config.workload.  Default workload = BASELINE.json configs[1]: the rollup circuit scaled to ~2^20
constraints (shape of BatchProcessTx(16, 6): 858 400 constraints, 577 public inputs, m = 2^20),
synthetic R1CS / witness / key (see simple_zk_rollups_b200/synth.py, keygen.py).
  value  proofs/s with the witness already resident in HBM (zkr_prove_dev), CUDA events on the launch stream
  e2e    proofs/s through the host API (zkr_prove_batch; zkr_prove per call is reported beside it): pinned-host
         witness H2D + proof D2H inside the timed region
N > 1 (torchrun, one rank per GPU): independent proofs, one per GPU, no data-path collective ("weak").
After the replica timing every run also measures, outside the headline timed region and reported as extra blocks:
  batch_2p22  BASELINE.json configs[4]: >= 8 independent ~2^22-constraint proofs per GPU through zkr_prove_batch
              (host witness buffers), every proof checked by zkr_verify
  sharded     (N > 1) SURVEY.md 8(e): one tx_2p20 proof split over the N GPUs (bytes == the 1-GPU proof on every
              rank), the four-step NTT at 2^24 / 2^26 with its all-to-all fused into a pass (closed-form check of
              transformed values + round trip), the G1 MSM at 2^24 sharded by point range (host-only expectation)
--impl reference: the C restatement of the reference's CPU algorithm (oracle/c, kind "port": the reference's
own prover is un-vendored JavaScript/WASM that cannot run in this image) on all host cores, rank 0 only.
ZKR_BENCH_ONE_DEVICE=1 (flow test on a 1-GPU box): all ranks share cuda:0 and torch.distributed runs on gloo.
--dump-outputs DIR: after the timed steps, the proof of the last timed step is written as DIR/proof.npy (rank k > 0:
proof_rank<k>.npy), see dump_proof.  Circuit, witness, key and (r, s) are seeded or fixed, so two builds run with the
same arguments can be compared output for output; both arms write the same file for the same workload.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOXIC = (0x1234567890ABCDEF1234567890ABCDEF1234567, 0x2222222222222222222222222222222222221,
         0x3333333333333333333333333333333333333331, 0x44444444444444444444444444444444441,
         0x555555555555555555555555555555555555555551)
BASELINE_CONFIG = {"tx": "BASELINE.json configs[0]", "tx_2p20": "BASELINE.json configs[1]",
                   "tx_2p22": "BASELINE.json configs[4] (per-GPU unit of the throughput batch)"}
MODMUL_IMAD = 136            # 8x8-limb CIOS: 128 wide MACs + 8 (SURVEY.md 8(d))
EXEC_IMAD_PER_MADD = 6 * 136 + 200 + 2 * 108   # what k_accum_affine<Fq> executes per mixed addition (DESIGN.md 4.3); algorithmic: 1360
MADD_MODMULS = 10            # XYZZ mixed add 8M + 2S
R_ORDER = 21888242871839275222246405745257275088548364400416034343698204186575808495617
Q_FIELD = 21888242871839275222246405745257275088696311157297823662689037894645226208583
RS = (0x1F2E3D4C5B6A79881122334455667788 << 64 | 0x99AABBCCDDEEFF00, 0x0123456789ABCDEF << 100 | 77)


def workload_string(shape, r1, n, bits):
    """config.workload, identical in both arms (the driver compares the strings)."""
    return ("BN254 Groth16 prove, rollup-shaped circuit %s: %d constraints, %d public, nVars %d, domain 2^%d; fixed (r,s)"
            % (shape, r1.nConstraints, r1.nPublic, n, bits))


def host_g1_mul(k):
    """k * G on BN254 G1 (G = (1, 2), y^2 = x^3 + 3), affine double-and-add on Python integers: the host-only
    expectation of the sharded MSM check.  -> 64 bytes x|y little-endian standard form (zeros = infinity)."""
    q = Q_FIELD

    def add(P, S):
        if P is None:
            return S
        if S is None:
            return P
        if P[0] == S[0]:
            if (P[1] + S[1]) % q == 0:
                return None
            lam = 3 * P[0] * P[0] * pow(2 * P[1], -1, q) % q
        else:
            lam = (S[1] - P[1]) * pow(S[0] - P[0], -1, q) % q
        x = (lam * lam - P[0] - S[0]) % q
        return x, (lam * (P[0] - x) - P[1]) % q

    acc, base = None, (1, 2)
    k %= R_ORDER
    while k:
        if k & 1:
            acc = add(acc, base)
        base = add(base, base)
        k >>= 1
    return bytes(64) if acc is None else acc[0].to_bytes(32, "little") + acc[1].to_bytes(32, "little")


def dot_mod_r(k_bytes, s_u64):
    """sum k_i * s_i mod r, exact (k: n x 32 B little-endian, s: n uint64): 16-bit-limb dot products in uint64."""
    import numpy as np
    n = s_u64.size
    k16 = k_bytes.view(np.uint16).reshape(n, 16).astype(np.uint64)
    s16 = s_u64.view(np.uint16).reshape(n, 4).astype(np.uint64)
    tot = 0
    for a in range(16):
        ka = k16[:, a]
        for b in range(4):
            acc = 0
            for lo in range(0, n, 1 << 26):           # partial sums stay < 2^63
                acc += int(np.dot(ka[lo:lo + (1 << 26)], s16[lo:lo + (1 << 26), b]))
            tot += acc << (16 * (a + b))
    return tot % R_ORDER


class DevView:
    """A raw device pointer as a torch uint8 tensor (torch is plumbing: compare / copy device buffers the library owns)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def dump_proof(out_dir, name, proof):
    """256 proof bytes (include/zkr.h: pi_a x|y, pi_b x.c0|x.c1|y.c0|y.c1, pi_c x|y) -> out_dir/<name>.npy, float64 of
    shape (8, 32): one coordinate per row, its 32 little-endian bytes as exact values 0..255."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    a = np.frombuffer(bytes(proof), dtype=np.uint8).reshape(8, 32).astype(np.float64)
    np.save(os.path.join(out_dir, name + ".npy"), a)


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(shape, seed):
    from simple_zk_rollups_b200 import synth
    nc, npub = synth.SHAPES[shape]
    t0 = time.time()
    r1, w = synth.generate(nc, npub, seed=seed)
    log("[bench] synthetic R1CS %s: %d constraints, %d public, nVars %d, nnz %s (%.1f s)" % (
        shape, nc, npub, r1.nVars, r1.nnz(), time.time() - t0))
    return r1, w


def run_ours(args):
    import numpy as np
    import torch
    from simple_zk_rollups_b200 import _lib, keygen, prover, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d" % (args.gpus, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libzkr has no CPU fallback")
    one_device = os.environ.get("ZKR_BENCH_ONE_DEVICE") == "1"     # flow test on a 1-GPU box: every rank on cuda:0, gloo
    if one_device:
        local = 0
        os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if one_device:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    red_dev = "cpu" if one_device else "cuda"
    L = _lib.lib()
    gp = prover.Groth16Prover(local)
    stream = torch.cuda.current_stream()
    _lib.check(L.zkr_ctx_set_stream(gp.ctx, C.c_void_p(stream.cuda_stream)))

    r1, w = make_workload(args.shape, seed=11 + rank)       # distinct witnesses per rank, same shape
    t0 = time.time()
    pk_bin, vk = keygen.synth_setup(gp.ctx, r1, TOXIC)
    key = gp.load_key(pk_bin)
    info = gp.key_info(key)
    log("[bench] key: %.1f MB binary, %.2f GB resident in HBM (%.1f s setup+load)" % (
        pk_bin.size / 1e6, info["device_bytes"] / 1e9, time.time() - t0))
    n, m = info["nVars"], info["domainSize"]
    wbytes = synth.witness_bytes(w)
    w_host = torch.frombuffer(bytearray(wbytes), dtype=torch.uint8).pin_memory()
    w_dev = w_host.cuda()
    proof_dev = torch.zeros(256, dtype=torch.uint8, device="cuda")
    rs = RS
    rb = np.frombuffer(int(rs[0]).to_bytes(32, "little"), dtype=np.uint8)
    sb = np.frombuffer(int(rs[1]).to_bytes(32, "little"), dtype=np.uint8)

    def prove_dev():
        _lib.check(L.zkr_prove_dev(gp.ctx, key, C.c_void_p(w_dev.data_ptr()), n, _lib.buf_ptr(rb), _lib.buf_ptr(sb),
                                   C.c_void_p(proof_dev.data_ptr())))

    out = np.zeros(256, dtype=np.uint8)
    stats = _lib.Stats()

    def prove_host():
        _lib.check(L.zkr_prove(gp.ctx, key, C.c_void_p(w_host.data_ptr()), n, _lib.buf_ptr(rb), _lib.buf_ptr(sb),
                               _lib.buf_ptr(out), C.byref(stats)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = gp.kernel_launches()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = gp.kernel_launches() - l0
        return max_over_ranks(ms), launches

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=red_dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(flag):
        if world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], device=red_dev, dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # parity guard: the proof must be what the host API returns for the same inputs
    prove_dev()
    torch.cuda.synchronize()
    prove_host()
    assert bytes(proof_dev.cpu().numpy().tobytes()) == out.tobytes(), "device and host API proofs differ"

    sampler = ClockSampler(local)
    sampler.start()
    ms, launches = timed(prove_dev, args.steps, args.warmup)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_proof(args.dump_outputs, "proof" if rank == 0 else "proof_rank%d" % rank, proof_dev.cpu().numpy())
    ms_e2e, _ = timed(prove_host, args.steps, max(args.warmup, 1))

    # e2e throughput through the batch entry point (the shape of many genTxVerifierProof calls): host witness
    # buffers, every proof's H2D and D2H inside the timed region, witness i+1 uploaded while proof i runs
    ctxs1, pks1 = (C.c_void_p * 1)(gp.ctx), (C.c_void_p * 1)(key)
    w_host2 = w_host.clone().pin_memory()
    rs_pair = np.concatenate([rb, sb])

    def prove_batch_host(nproofs):
        wptrs = (C.c_void_p * nproofs)(*[(w_host if i % 2 == 0 else w_host2).data_ptr() for i in range(nproofs)])
        rsb = np.tile(rs_pair, nproofs)
        outb = np.zeros(256 * nproofs, dtype=np.uint8)
        _lib.check(L.zkr_prove_batch(ctxs1, pks1, 1, wptrs, n, nproofs, _lib.buf_ptr(rsb), _lib.buf_ptr(outb)))
        return outb

    ob = prove_batch_host(max(args.warmup, 2))
    assert ob[-256:].tobytes() == out.tobytes(), "batch and single-call proofs differ"
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    ob = prove_batch_host(args.steps)
    e1.record(stream)
    barrier()
    ms_batch = e0.elapsed_time(e1)
    assert ob[-256:].tobytes() == out.tobytes() and ob[:256].tobytes() == out.tobytes()
    ms_batch = max_over_ranks(ms_batch)
    # the same call with TWO contexts (and key replicas) on this GPU: zkr_prove_batch deals the proofs round-robin, so two
    # proofs are in flight and one proof's latency-bound tail overlaps the other's bulk kernels
    ms_batch2 = None
    if not args.no_two_in_flight:
        K = max(2, args.in_flight)
        extra, streams, keys_k = [], [], []
        for _ in range(K - 1):
            g2_ = prover.Groth16Prover(local)
            st_ = torch.cuda.Stream()
            _lib.check(L.zkr_ctx_set_stream(g2_.ctx, C.c_void_p(st_.cuda_stream)))
            extra.append(g2_)
            streams.append(st_)
            keys_k.append(g2_.load_key(pk_bin))
        ctxs2 = (C.c_void_p * K)(gp.ctx, *[e_.ctx for e_ in extra])
        pks2 = (C.c_void_p * K)(key, *keys_k)

        def prove_batch_host2(nproofs):
            wptrs = (C.c_void_p * nproofs)(*[(w_host if i % 2 == 0 else w_host2).data_ptr() for i in range(nproofs)])
            rsb = np.tile(rs_pair, nproofs)
            outb = np.zeros(256 * nproofs, dtype=np.uint8)
            _lib.check(L.zkr_prove_batch(ctxs2, pks2, K, wptrs, n, nproofs, _lib.buf_ptr(rsb), _lib.buf_ptr(outb)))
            return outb
        ob = prove_batch_host2(2 * K)
        assert all(ob[256 * i:256 * i + 256].tobytes() == out.tobytes() for i in range(2 * K)), "in-flight proofs differ"
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ob = prove_batch_host2(K * args.steps)
        e1.record(stream)
        barrier()
        ms_batch2 = max_over_ranks(e0.elapsed_time(e1)) / K            # per `steps` proofs, comparable with ms_batch
        assert all(ob[256 * i:256 * i + 256].tobytes() == out.tobytes() for i in range(K * args.steps))
        for e_ in extra:
            e_.close()
    _lib.check(L.zkr_prove_check(gp.ctx, key))       # input-validity flags of the zkr_prove_dev calls above
    stage_ms = {k: round(v, 3) for k, v in stats.as_dict().items() if k.endswith("_ms")}
    ms_single_gpu_proof = ms_e2e / args.steps

    # ---- SURVEY 8(f) rank 4: the witness made on the GPU (forward solve of the circuit) and proved where it lies
    gpu_witness = None
    if not args.no_gpu_witness:
        from simple_zk_rollups_b200 import witness as wmod
        t0 = time.time()
        ws = wmod.WitnessSolver(gp, r1)
        t_build = time.time() - t0
        given = ws.given_from_witness(w)
        gbuf = np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in given), dtype=np.uint8)
        proof_dev2 = torch.zeros(256, dtype=torch.uint8, device="cuda")

        def solve_only():
            _lib.check(L.zkr_witness_solve(gp.ctx, ws.h, _lib.buf_ptr(gbuf), ws.d_witness))

        def solve_and_prove():
            solve_only()
            _lib.check(L.zkr_prove_dev(gp.ctx, key, ws.d_witness, n, _lib.buf_ptr(rb), _lib.buf_ptr(sb),
                                       C.c_void_p(proof_dev2.data_ptr())))
        solve_and_prove()
        torch.cuda.synchronize()
        _lib.check(L.zkr_prove_check(gp.ctx, key))
        same = bytes(proof_dev2.cpu().numpy().tobytes()) == out.tobytes()
        ms_solve, _ = timed(solve_only, args.steps, 1)
        ms_sp, _ = timed(solve_and_prove, args.steps, 1)
        gpu_witness = {"what": "zkr_witness_solve (forward solve of the circuit on the GPU from its given signals) + zkr_prove_dev on the "
                               "resident witness: createProofGenerator without the host-side witness calculator's bulk",
                       "given_signals": ws.n_given, "solved_signals": ws.n_solved, "levels": ws.n_levels,
                       "build_s": round(t_build, 2), "h2d_bytes_per_proof": 32 * ws.n_given + 64,
                       "solve_ms": round(ms_solve / args.steps, 4), "solve_plus_prove_ms": round(ms_sp / args.steps, 4),
                       "proofs_per_s": round(world * args.steps / (ms_sp * 1e-3), 3),
                       "proof_identical_to_host_witness_proof": bool(all_true(same))}
        ws.close()

    # ---- extra blocks (outside the headline timed region): sharded paths of SURVEY 8(e), config 5 batch
    env = dict(torch=torch, dist=dist, L=L, gp=gp, stream=stream, rank=rank, world=world, local=local,
               barrier=barrier, max_over_ranks=max_over_ranks, all_true=all_true, red_dev=red_dev)
    sharded = None
    if world > 1 and not args.no_sharded:
        sharded = sharded_blocks(env, args, key_rank0=(key, pk_bin, wbytes, out.tobytes(), ms_single_gpu_proof))
    batch_2p22 = None
    if not args.no_batch_2p22 and args.shape == "tx_2p20":
        batch_2p22 = batch_block(env, args, "tx_2p22", 8)

    result = None
    if rank == 0:
        # ---- roofline of the dominant kernel (G1 bucket accumulation), measured live on a serialised pass
        _lib.check(L.zkr_ctx_set_serial(gp.ctx, 1))
        _lib.check(L.zkr_ctx_set_profile(gp.ctx, 1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        prof_steps = min(args.steps, 4)
        e0.record(stream)
        for _ in range(prof_steps):
            prove_dev()
        e1.record(stream)
        torch.cuda.synchronize()
        serial_ms = e0.elapsed_time(e1) / prof_steps
        prof = {}
        for pid, name in ((0, "accum_g1"), (1, "accum_g2"), (2, "ntt_pass")):
            tot, cnt, units = C.c_double(), C.c_int(), C.c_double()
            _lib.check(L.zkr_ctx_profile_read(gp.ctx, pid, C.byref(tot), C.byref(cnt), C.byref(units)))
            prof[name] = (tot.value, cnt.value, units.value)
        _lib.check(L.zkr_ctx_set_profile(gp.ctx, 0))
        _lib.check(L.zkr_ctx_set_serial(gp.ctx, 0))
        imad_peak, ms_mb = C.c_double(), C.c_float()
        _lib.check(L.zkr_microbench(gp.ctx, 0, 100000, C.byref(imad_peak), C.byref(ms_mb)))
        modmul_peak = C.c_double()
        _lib.check(L.zkr_microbench(gp.ctx, 2, 20000, C.byref(modmul_peak), C.byref(ms_mb)))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            pass
        g1_ms, g1_cnt, g1_madds = prof["accum_g1"]
        roofline = None
        if g1_cnt:
            imads = g1_madds * MADD_MODMULS * MODMUL_IMAD
            ach = imads / (g1_ms * 1e-3) / 1e12
            roofline = {"kernel": "k_accum_affine<Fq> (G1 bucket accumulation, XYZZ mixed adds)",
                        "bound": "imad", "achieved": round(ach, 3), "peak": round(imad_peak.value / 1e12, 3),
                        "unit": "TIMAD/s", "frac": round(ach / (imad_peak.value / 1e12), 4),
                        "traffic": traffic.get("accum_g1_bytes_per_launch"),
                        "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu "
                                          "--set full capture (profiles/ncu_traffic.json), NOT measured in this run",
                        "peak_source": "plain IMAD chain measured in this run (zkr_microbench); MEASURED_PEAKS.json has no integer peak",
                        "practical_peak_frac": round((g1_madds * MADD_MODMULS / (g1_ms * 1e-3)) / modmul_peak.value, 4),
                        "practical_peak_note": "vs the register-resident Fq modmul chain measured in this run (%.1f G modmul/s): "
                                               "IMAD.WIDE issues at half the IMAD rate.  The count is the ALGORITHMIC 10 modmul per "
                                               "mixed addition (SURVEY.md 8(d)); since round 2 the kernel executes 1232 IMAD per "
                                               "addition instead of 1360 (y3 = r (q - x3) - y ppp as one two-product pass with one "
                                               "reduction: 200 instead of 272; the two squarings with every cross product taken once: 108 "
                                               "instead of 136 each), which is how this fraction can exceed the chain's" % (modmul_peak.value / 1e9),
                        "executed_imad_per_madd": EXEC_IMAD_PER_MADD,
                        "executed_frac_of_plain_imad_peak": round(g1_madds * EXEC_IMAD_PER_MADD / (g1_ms * 1e-3) / imad_peak.value, 4),
                        "launches": g1_cnt, "avg_launch_ms": round(g1_ms / g1_cnt, 4),
                        "algorithmic_units_per_launch": "%.0f mixed adds x 10 modmul x 136 IMAD" % (g1_madds / g1_cnt),
                        "share_of_serial_step": round(g1_ms / prof_steps / serial_ms, 4),
                        "measured": "serialised pass of the same step (zkr_ctx_set_serial), CUDA events on the launch stream"}
        nt_ms, nt_cnt, nt_elems = prof["ntt_pass"]
        roofline_ntt = None
        if nt_cnt:
            gbs = 64.0 * nt_elems / (nt_ms * 1e-3) / 1e9
            roofline_ntt = {"kernel": "k_ntt_pass (one <=11-bit radix pass over 2^%d Fr elements)" % (m.bit_length() - 1),
                            "bound": "hbm", "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                            "frac": round(gbs / hbm_peak, 4), "traffic": traffic.get("ntt_pass_bytes_per_launch"),
                            "traffic_source": "static (profiles/ncu_traffic.json), not measured in this run",
                            "peak_source": hbm_src, "launches": nt_cnt, "avg_launch_ms": round(nt_ms / nt_cnt, 4),
                            "note": "64 B per element per pass (read once + write once); the pass is IMAD-bound "
                                    "(~6 modmul per 64 B), see DESIGN.md"}
            # the binding roof (SURVEY 8(d)): butterfly modmuls, (m/2) log2 m per transform, 6 transforms per proof
            log_m = m.bit_length() - 1
            bfly = 6.0 * prof_steps * (m // 2) * log_m
            roofline_ntt["imad"] = {
                "bound": "imad", "butterfly_modmuls_per_proof": int(bfly / prof_steps),
                "achieved_timad_per_s": round(bfly * MODMUL_IMAD / (nt_ms * 1e-3) / 1e12, 3),
                "frac_of_plain_imad_peak": round(bfly * MODMUL_IMAD / (nt_ms * 1e-3) / imad_peak.value, 4),
                "frac_of_practical_modmul_peak": round(bfly / (nt_ms * 1e-3) / modmul_peak.value, 4),
                "note": "algorithmic butterflies only; the passes of a proof also carry the fused element-wise work (A.B products, "
                        "coset scaling, h assembly) and the inter-pass twiddles, which are not counted: see `transform` for a bare "
                        "transform and `h_pipeline` for the whole pipeline against its algorithmic count"}
        if roofline_ntt is not None:
            # standalone figures of the same size (data resident, kernel-only, best of 10): one forward transform -- the
            # "NTT GB/s" of BASELINE.json's metric -- and the whole H pipeline (6 transforms, element-wise work fused into
            # their passes) against SURVEY 8(d)'s algorithmic count 7 NTT(m) + 3 m modmuls
            log_m = m.bit_length() - 1
            bufs = [torch.randint(0, 256, (m * 32,), dtype=torch.uint8, device="cuda") for _ in range(3)]
            for b_ in bufs:
                b_.view(m, 32)[:, 31] &= 0x1F

            def best10(fn):
                fn()
                torch.cuda.synchronize()
                best = 1e30
                for _ in range(10):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    fn()
                    e1.record(stream)
                    torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1))
                return best
            t_fwd = best10(lambda: _lib.check(L.zkr_ntt(gp.ctx, C.c_void_p(bufs[0].data_ptr()), log_m, 0 | 0x10, 1)))
            t_h = best10(lambda: _lib.check(L.zkr_h_from_evals_dev(gp.ctx, C.c_void_p(bufs[0].data_ptr()), C.c_void_p(bufs[1].data_ptr()),
                                                                   log_m, C.c_void_p(bufs[2].data_ptr()), 1)))
            bf1 = (m // 2) * log_m
            roofline_ntt["transform"] = {
                "what": "one forward DIF transform of 2^%d elements (zkr_ntt, natural in, bit-reversed out)" % log_m,
                "ms": round(t_fwd, 4), "gb_per_s": round(64.0 * m / (t_fwd * 1e-3) / 1e9, 1),
                "hbm_frac": round(64.0 * m / (t_fwd * 1e-3) / 1e9 / hbm_peak, 4),
                "frac_of_plain_imad_peak": round(bf1 * MODMUL_IMAD / (t_fwd * 1e-3) / imad_peak.value, 4),
                "frac_of_practical_modmul_peak": round(bf1 / (t_fwd * 1e-3) / modmul_peak.value, 4)}
            hm = 7 * bf1 + 3 * m
            roofline_ntt["h_pipeline"] = {
                "what": "A_T, B_T -> h (zkr_h_from_evals_dev): 6 transforms, no separate element-wise sweep",
                "ms": round(t_h, 4), "algorithmic_modmuls": hm,
                "frac_of_plain_imad_peak": round(hm * MODMUL_IMAD / (t_h * 1e-3) / imad_peak.value, 4),
                "frac_of_practical_modmul_peak": round(hm / (t_h * 1e-3) / modmul_peak.value, 4)}
            del bufs
        # ---- CPU baseline: the C restatement of the reference algorithm on this box's host cores
        cpu = None if args.no_cpu else cpu_baseline(pk_bin, wbytes, rs, out.tobytes(), args)
        value = world * args.steps / (ms * 1e-3)
        e2e_one = world * args.steps / (ms_batch * 1e-3)
        e2e_two = world * args.steps / (ms_batch2 * 1e-3) if ms_batch2 else None
        use_two = e2e_two is not None and e2e_two > e2e_one
        e2e_val = e2e_two if use_two else e2e_one
        ms_e2e_step = (ms_batch2 if use_two else ms_batch) / args.steps
        result = {
            "metric": "groth16_proofs_per_s", "value": round(value, 3), "unit": "proofs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (8x32-bit-limb Montgomery, integer pipe)",
            "data": "synthetic",
            "config": {"workload": workload_string(args.shape, r1, n, m.bit_length() - 1),
                       "key_resident_in_hbm": True,
                       "baseline_config": BASELINE_CONFIG.get(args.shape, "BASELINE.json configs[1] shape family"),
                       "parallelism": "one independent proof per GPU",
                       "l2": "per-proof working set (%.1f GB of window tables + sort buffers) >> 126 MB L2; no flush needed" % (
                           info["device_bytes"] / 1e9)},
            "prove_ms": round(ms / args.steps, 4), "prove_ms_e2e": round(ms_e2e / args.steps, 4),
            "prove_ms_serial": round(serial_ms, 4),
            "e2e": {"value": round(e2e_val, 3), "unit": "proofs/s", "h2d_bytes_per_step": 32 * n + 64,
                    "d2h_bytes_per_step": 256, "ms_per_step": round(ms_e2e_step, 4),
                    "api": "zkr_prove_batch on host witness buffers (pinned): per proof H2D of the witness + (r,s), "
                           "D2H of the 256-byte proof and the range flags; witness i+1 is uploaded while proof i runs"
                           + ("; %d contexts with one key replica each per GPU = %d proofs in flight" % (max(2, args.in_flight), max(2, args.in_flight)) if use_two else
                              "; one context per GPU = one proof in flight"),
                    "one_in_flight": {"value": round(e2e_one, 3), "ms_per_step": round(ms_batch / args.steps, 4)},
                    "two_in_flight": None if e2e_two is None else {"value": round(e2e_two, 3), "ms_per_step": round(ms_batch2 / args.steps, 4),
                                                                   "key_replicas_per_gpu": max(2, args.in_flight)},
                    "single_call": {"api": "zkr_prove (one blocking call per proof, nothing overlapped)",
                                    "value": round(world * args.steps / (ms_e2e * 1e-3), 3),
                                    "ms_per_step": round(ms_e2e / args.steps, 4)}},
            "gpu_launches": int(launches), "clocks": clocks, "stage_ms_overlapped": stage_ms,
            "roofline": roofline, "roofline_ntt": roofline_ntt, "cpu_baseline": cpu,
            "gpu_witness": gpu_witness, "batch_2p22": batch_2p22, "sharded": sharded,
        }
    gp.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if result is not None:
        print(json.dumps(result), flush=True)


def best_of(env, fn, reps):
    """best-of-reps device time of fn (ms): barrier, CUDA events on the launch stream, max over ranks per rep."""
    torch, stream = env["torch"], env["stream"]
    fn()
    best = 1e30
    for _ in range(reps):
        env["barrier"]()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        best = min(best, env["max_over_ranks"](e0.elapsed_time(e1)))
    return best


def batch_block(env, args, shape, per_gpu):
    """BASELINE.json configs[4]: independent ~2^22-constraint proofs, one in flight per GPU, through zkr_prove_batch with
    HOST witness buffers (H2D of every witness and D2H of every proof inside the timed region).  Each rank makes its own
    circuit + key (seeded) and two distinct witnesses of it, proves `per_gpu` proofs with distinct (r, s), and checks
    every one with the library's verifier (zkr_verify: GPU vk_x MSM + host pairing product)."""
    import numpy as np
    from simple_zk_rollups_b200 import keygen, synth
    torch, L, gp, rank, world = env["torch"], env["L"], env["gp"], env["rank"], env["world"]
    nc, npub = synth.SHAPES[shape]
    t0 = time.time()
    r1, w0 = synth.generate(nc, npub, seed=41 + rank, witness_seed=1)
    _, w1 = synth.generate(nc, npub, seed=41 + rank, witness_seed=2)
    assert w0[1:8] != w1[1:8]
    t1 = time.time()
    pk_bin, vk = keygen.synth_setup(gp.ctx, r1, TOXIC)
    key = gp.load_key(pk_bin)
    vkey = gp.load_vkey(vk["bin"])
    info = gp.key_info(key)
    n = info["nVars"]
    log("[bench] %s: %d constraints, nVars %d, 2 witnesses %.1f s, setup + load %.1f s, %.1f GB resident" % (
        shape, nc, n, t1 - t0, time.time() - t1, info["device_bytes"] / 1e9))
    wh = [torch.frombuffer(bytearray(synth.witness_bytes(w)), dtype=torch.uint8).pin_memory() for w in (w0, w1)]
    pubs = [w[1:npub + 1] for w in (w0, w1)]
    ctxs1, pks1 = (C.c_void_p * 1)(gp.ctx), (C.c_void_p * 1)(key)
    import random
    rng = random.Random(1000 + rank)

    def run(nproofs):
        wptrs = (C.c_void_p * nproofs)(*[wh[i % 2].data_ptr() for i in range(nproofs)])
        rsb = np.frombuffer(b"".join(rng.randrange(R_ORDER).to_bytes(32, "little") for _ in range(2 * nproofs)), dtype=np.uint8)
        outb = np.zeros(256 * nproofs, dtype=np.uint8)
        _lib_check(L.zkr_prove_batch(ctxs1, pks1, 1, wptrs, n, nproofs, _buf_ptr(rsb), _buf_ptr(outb)))
        return outb

    run(2)                                            # warm-up
    env["barrier"]()
    stream = env["stream"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    outb = run(per_gpu)
    e1.record(stream)
    env["barrier"]()
    ms = env["max_over_ranks"](e0.elapsed_time(e1))
    ok = len({outb[256 * i:256 * i + 256].tobytes() for i in range(per_gpu)}) == per_gpu       # distinct proofs
    for i in range(per_gpu):
        ok = ok and gp.verify(vkey, outb[256 * i:256 * i + 256].tobytes(), pubs[i % 2])
    ok = env["all_true"](ok)
    gp.L.zkr_pkey_free(key)
    gp._keys.remove(key)
    total = per_gpu * world
    return {"baseline_config": "BASELINE.json configs[4]", "shape": shape, "constraints": nc, "domain_log2": (info["domainSize"]).bit_length() - 1,
            "proofs": total, "proofs_per_gpu": per_gpu, "n_gpus": world, "ms": round(ms, 3),
            "proofs_per_s": round(total / (ms * 1e-3), 3), "ms_per_proof_per_gpu": round(ms / per_gpu, 3),
            "key_gb_per_gpu": round(info["device_bytes"] / 1e9, 2), "h2d_bytes_per_proof": 32 * n + 64, "d2h_bytes_per_proof": 256,
            "api": "zkr_prove_batch, host witness buffers (pinned), witness i+1 uploaded while proof i runs",
            "witnesses": "2 distinct witnesses per GPU (distinct seeds), distinct (r, s) per proof, one key per GPU",
            "all_proofs_verify": bool(ok), "identical": bool(ok),
            "check": "every proof accepted by zkr_verify (TxVerifier.sol:258-276 predicate) for its own public inputs; proofs pairwise distinct"}


def sharded_blocks(env, args, key_rank0):
    """SURVEY.md 8(e) on N GPUs over peer memory (csrc/comm.cu), every result checked:
       proof  zkr_prove_sharded on the tx_2p20 key of rank 0's replica run: 256 bytes == rank 0's 1-GPU proof on every rank
       ntt    zkr_ntt_sharded 2^24 / 2^26, input x_j = c g^j: transformed values at 8 random + first / last local positions
              against the closed form c (g^N - 1) / (g w^k - 1) on Python ints, and DIT^-1(DIF(x)) == x on the whole slab
       msm    zkr_msm_sharded G1 2^24, P_i = s_i G: result == (sum k_i s_i mod r) G with the sum and the scalar
              multiplication done on the host (numpy + Python ints)"""
    import numpy as np
    from simple_zk_rollups_b200 import keygen, sharding as sh, synth
    torch, dist, L, gp = env["torch"], env["dist"], env["L"], env["gp"]
    rank, world, stream = env["rank"], env["world"], env["stream"]
    red_dev = env["red_dev"]
    ctx = gp.ctx
    reps = 5
    ntt_logs = [int(v) for v in args.sharded_ntt_logs.split(",") if v]
    msm_logs = [int(v) for v in str(args.sharded_msm_log).split(",") if v]
    comm = sh.Comm(ctx, rank, world, (1 << max(ntt_logs + [16])) // world)
    comm.connect_torch()
    res = {"n_gpus": world, "transport": "peer memory over NVLink (CUDA IPC mapped slabs, remote stores from the producing kernels, "
                                         "device-side flag barrier); torch.distributed only swaps the 64-byte IPC handles"}

    def bcast_bytes(b, n):
        t = torch.frombuffer(bytearray(b if rank == 0 else bytes(n)), dtype=torch.uint8).to(red_dev)
        dist.broadcast(t, 0)
        return t.cpu().numpy().tobytes()

    # ------------------------------------------------------------------ one proof over N GPUs
    key0, pk_bin0, wbytes0, proof0, single_ms = key_rank0
    t0 = time.time()
    if rank == 0:
        pk_bin, wbytes = pk_bin0, wbytes0
    else:                                             # same circuit / witness / key as rank 0 (seeded generators)
        nc, npub = synth.SHAPES[args.shape]
        r1, w = synth.generate(nc, npub, seed=11)
        pk_bin, _ = keygen.synth_setup(ctx, r1, TOXIC)
        wbytes = synth.witness_bytes(w)
    part = gp.load_key_sharded(pk_bin, rank, world)
    want = bcast_bytes(proof0, 256)
    single_ms = env["max_over_ranks"](single_ms if rank == 0 else 0.0)
    # pinned, like the witness buffer of the one-GPU call it is compared with
    wit_pin = torch.frombuffer(bytearray(wbytes), dtype=torch.uint8).pin_memory()
    rb = np.frombuffer(int(RS[0]).to_bytes(32, "little"), dtype=np.uint8)
    sb = np.frombuffer(int(RS[1]).to_bytes(32, "little"), dtype=np.uint8)
    got = np.zeros(256, dtype=np.uint8)
    st = _Stats()

    def prove_sharded():
        _lib_check(L.zkr_prove_sharded(comm.h, part, C.c_void_p(wit_pin.data_ptr()), wit_pin.numel() // 32, _buf_ptr(rb), _buf_ptr(sb),
                                       _buf_ptr(got), C.byref(st)))
    t_sh = best_of(env, prove_sharded, reps)
    same = env["all_true"](got.tobytes() == want)
    info = gp.key_info(part)
    res["proof"] = {
        "shape": args.shape, "api": "zkr_pkey_load_bin_sharded + zkr_prove_sharded (pinned host witness, H2D + D2H inside)",
        "ms": round(t_sh, 3), "single_gpu_ms": round(single_ms, 3), "speedup_vs_1gpu": round(single_ms / t_sh, 3),
        "identical": bool(same), "check": "256 proof bytes on every rank == rank 0's zkr_prove on one GPU (same key, witness, r, s)",
        "exchange_bytes_per_rank": 1024 * (world - 1), "key_gb_per_rank": round(info["device_bytes"] / 1e9, 2),
        "stage_ms": {k: round(v, 3) for k, v in st.as_dict().items() if k.endswith("_ms")},
        "split": "task-aware (DESIGN.md 6): sparse LC + H pipeline + hExps MSM on the first max(1, N/2) ranks only, the witness MSMs' "
                 "point ranges weighted so that every rank carries the same modelled work; ZKR_SHARD_TASKS=0 = uniform ranges, H on every rank",
        "limited_by": "the 0.55 ms witness upload every rank repeats, the H chain (LC + 6 transforms + MSM, about 5 ms at 2^20) that bounds "
                      "its group however few witness points it also takes, and per-MSM latency chains (sort passes, gather, bucket "
                      "reduction, blinding: about 1.5 ms) that do not shrink with the point range (DESIGN.md 6)"}
    log("[bench] sharded proof: %.2f ms on %d GPUs vs %.2f ms on one, identical=%s (%.1f s)" % (
        t_sh, world, single_ms, same, time.time() - t0))
    gp.L.zkr_pkey_free(part)
    gp._keys.remove(part)

    # ------------------------------------------------------------------ four-step NTT, all-to-all fused into a pass
    cval, gval = 0x1234567890ABCDEF1234567890ABCDEF0F1E2D3C4B5A6978 % R_ORDER, 0x0FEDCBA9876543210FEDCBA987654321 % R_ORDER
    cb = np.frombuffer(cval.to_bytes(32, "little"), dtype=np.uint8)
    gb = np.frombuffer(gval.to_bytes(32, "little"), dtype=np.uint8)
    res["ntt"] = []
    for lg in ntt_logs:
        t0 = time.time()
        n = 1 << lg
        nl = n // world
        if lg - (world.bit_length() - 1) < 11:        # csrc/ntt.cu ntt_run_sharded: every rank needs at least one full 2^11 tile row
            res["ntt"].append({"log_n": lg, "skipped": "2^%d over %d ranks is below the sharded transform's minimum tile geometry" % (lg, world),
                               "identical": True})
            continue
        w = pow(5, (R_ORDER - 1) >> lg, R_ORDER)
        top = cval * (pow(gval, n, R_ORDER) - 1) % R_ORDER

        def closed(k):
            return top * pow((gval * pow(w, k, R_ORDER) - 1) % R_ORDER, -1, R_ORDER) % R_ORDER

        def brev(x):
            return int(bin(x)[2:].zfill(lg)[::-1], 2)

        def fill(dst_ptr, wd, rk):
            _lib_check(L.zkr_fill_geometric(ctx, C.c_void_p(dst_ptr), n // wd, _buf_ptr(cb), _buf_ptr(gb), 0, lg, wd, rk))
        import random
        rng = random.Random(77 * lg + rank)
        probes = [0, nl - 1] + [rng.randrange(nl) for _ in range(8)]
        # single-GPU transform of the same vector on every rank's own GPU (baseline + closed-form check)
        single = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        fill(single.data_ptr(), 1, 0)
        _lib_check(L.zkr_ntt(ctx, C.c_void_p(single.data_ptr()), lg, sh.NTT_FORWARD | sh.NTT_BITREV_OUT, 1))
        torch.cuda.synchronize()
        ok1 = True
        for p_ in probes[:4]:
            pos = rank * nl + p_
            v = int.from_bytes(single[32 * pos:32 * pos + 32].cpu().numpy().tobytes(), "little")
            ok1 = ok1 and v == closed(brev(pos))
        t_single = best_of(env, lambda: _lib_check(L.zkr_ntt(ctx, C.c_void_p(single.data_ptr()), lg,
                                                             sh.NTT_FORWARD | sh.NTT_BITREV_OUT, 1)), reps)
        del single
        # sharded: COLS slab in buffer 0 -> DIF -> ROWS slab (bit-reversed order) in buffer 1
        fill(comm.buffer(0), world, rank)
        comm.ntt(lg, sh.NTT_FORWARD | sh.NTT_BITREV_OUT, 0)
        torch.cuda.synchronize()
        comm.check()
        rows = torch.as_tensor(DevView(comm.buffer(1), nl * 32), device="cuda")
        ok2 = True
        for p_ in probes:
            v = int.from_bytes(rows[32 * p_:32 * p_ + 32].cpu().numpy().tobytes(), "little")
            ok2 = ok2 and v == closed(brev(rank * nl + p_))
        # chain back: DIT inverse of the ROWS data must return the COLS slab of x, every byte
        comm.ntt(lg, sh.NTT_INVERSE | sh.NTT_BITREV_IN, 1)
        torch.cuda.synchronize()
        comm.check()
        ref = torch.empty(nl * 32, dtype=torch.uint8, device="cuda")
        fill(ref.data_ptr(), world, rank)
        torch.cuda.synchronize()
        ok3 = bool(torch.equal(ref, torch.as_tensor(DevView(comm.buffer(0), nl * 32), device="cuda")))
        del ref
        _lib_check(L.zkr_ctx_set_profile(ctx, 1))
        t_dif = best_of(env, lambda: comm.ntt(lg, sh.NTT_FORWARD | sh.NTT_BITREV_OUT, 0), reps)
        xt, xc, xu = C.c_double(), C.c_int(), C.c_double()
        _lib_check(L.zkr_ctx_profile_read(ctx, 3, C.byref(xt), C.byref(xc), C.byref(xu)))
        _lib_check(L.zkr_ctx_set_profile(ctx, 0))
        t_dit = best_of(env, lambda: comm.ntt(lg, sh.NTT_INVERSE | sh.NTT_BITREV_IN, 1), reps)
        comm.check()
        xpass_ms = env["max_over_ranks"](xt.value / max(xc.value, 1))
        xbytes = 32 * nl * (world - 1) // world
        row = {"log_n": lg, "dif_ms": round(t_dif, 4), "dit_inverse_ms": round(t_dit, 4), "single_gpu_dif_ms": round(t_single, 4),
               "speedup_vs_1gpu": round(t_single / t_dif, 3), "aggregate_gb_per_s": round(64.0 * n / (t_dif * 1e-3) / 1e9, 1),
               "exchange_bytes_per_rank": xbytes, "exchange_pass_ms": round(xpass_ms, 4),
               "nvlink_gb_per_s_per_rank": round(xbytes / (xpass_ms * 1e-3) / 1e9, 1),
               "nvlink_note": "bytes this rank stores into its peers' HBM / duration of the pass whose write-back is the exchange "
                              "(the pass also computes its butterflies, so this is a lower bound on link throughput)",
               "values_checked": len(probes), "roundtrip_identical": ok3,
               "identical": bool(env["all_true"](ok1 and ok2 and ok3)),
               "check": "x_j = c g^j: transformed values (8 random + first + last local position per rank) == c (g^N - 1) / (g w^k - 1) on "
                        "Python ints, single-GPU and sharded; DIT^-1(DIF(x)) == x over the whole slab",
               "limited_by": "the exchange pass is the IMAD-bound column pass plus remote stores; barriers are two flag kernels"}
        res["ntt"].append(row)
        log("[bench] sharded NTT 2^%d: dif %.3f ms (1 GPU %.3f), identical=%s (%.1f s)" % (lg, t_dif, t_single, row["identical"], time.time() - t0))

    # ------------------------------------------------------------------ G1 MSM sharded by point range
    res["msm_g1"] = []
    for msm_log in msm_logs:
        t0 = time.time()
        n = 1 << msm_log
        chunks = 8                                        # generator granularity: the same vectors for every world size
        cn = n // chunks

        def chunk(j):
            g_ = np.random.default_rng(5000 + 16 * msm_log + j)
            s64 = g_.integers(1, 1 << 63, size=cn, dtype=np.uint64)
            k = g_.integers(0, 256, size=(cn, 32), dtype=np.uint8)
            k[:, 31] &= 0x1F                              # < 2^253 < r
            sel = g_.random(cn) < 0.03                    # rollup-like: 3 % of the scalars in {0, 1}
            k[sel] = 0
            k[sel, 0] = g_.integers(0, 2, size=int(sel.sum()), dtype=np.uint8)
            return s64, k

        def make_bases(lo, hi):
            js = range(lo // cn, hi // cn)
            parts = [chunk(j) for j in js]
            s64 = np.concatenate([p_[0] for p_ in parts])
            k = np.concatenate([p_[1] for p_ in parts])
            sc = np.zeros((hi - lo, 32), dtype=np.uint8)
            sc[:, :8] = s64.view(np.uint8).reshape(hi - lo, 8)
            pts = np.empty((hi - lo) * 64, dtype=np.uint8)
            _lib_check(L.zkr_synth_points(ctx, 1, _buf_ptr(sc), hi - lo, _buf_ptr(pts)))
            bases = C.c_void_p()
            _lib_check(L.zkr_bases_load(ctx, 1, _buf_ptr(pts), hi - lo, 0, C.byref(bases)))
            d_k = torch.from_numpy(np.ascontiguousarray(k).reshape(-1)).cuda()
            return bases, d_k, s64, k

        lo, hi = rank * (n // world), (rank + 1) * (n // world)
        bases, d_k, s64, k = make_bases(lo, hi)
        e_part = dot_mod_r(k.reshape(-1), s64)            # this rank's share of sum k_i s_i, on the host
        outp = comm.msm(bases, d_k.data_ptr(), hi - lo, on_device=True)[:64].tobytes()
        t_msm = best_of(env, lambda: comm.msm(bases, d_k.data_ptr(), hi - lo, on_device=True), reps)
        cc, ww = C.c_int(), C.c_int()
        _lib_check(L.zkr_bases_info(bases, None, C.byref(cc), C.byref(ww), None))
        L.zkr_bases_free(bases)
        del d_k
        parts = [None] * world
        dist.all_gather_object(parts, (int(e_part), outp))
        e = sum(p_[0] for p_ in parts) % R_ORDER
        ok = all(p_[1] == parts[0][1] for p_ in parts) and outp == host_g1_mul(e)
        # single-GPU baseline on rank 0 (the other ranks wait)
        t_single = 0.0
        if rank == 0:
            b1, dk1, s1, k1 = make_bases(0, n)
            o1 = np.zeros(64, dtype=np.uint8)
            _lib_check(L.zkr_msm(ctx, b1, C.c_void_p(dk1.data_ptr()), n, 1, _buf_ptr(o1)))
            ok = ok and o1.tobytes() == outp
            d_out = torch.zeros(256, dtype=torch.uint8, device="cuda")
            fn = lambda: _lib_check(L.zkr_msm_dev(ctx, b1, C.c_void_p(dk1.data_ptr()), n, C.c_void_p(d_out.data_ptr())))
            fn()
            torch.cuda.synchronize()
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                torch.cuda.synchronize()
                t_single = e0.elapsed_time(e1) if t_single == 0.0 else min(t_single, e0.elapsed_time(e1))
            L.zkr_bases_free(b1)
            del dk1
        t_single = env["max_over_ranks"](t_single)
        row = {"log_n": msm_log, "ms": round(t_msm, 4), "single_gpu_ms": round(t_single, 4),
                         "speedup_vs_1gpu": round(t_single / t_msm, 3), "gpts_per_s": round(n / t_msm / 1e6, 4),
                         "window_bits_per_rank": cc.value, "windows": ww.value, "exchange_bytes_per_rank": 128 * (world - 1),
                         "identical": bool(env["all_true"](ok)),
                         "check": "P_i = s_i G (64-bit s_i), rollup-like scalars: every rank's result == (sum k_i s_i mod r) G with the sum "
                                  "(numpy 16-bit-limb dot products) and the scalar multiplication (Python ints) on the host; == the 1-GPU MSM",
                         "limited_by": "fixed per-MSM latency (radix-sort passes, boundary levels, bucket reduction) at 2^%d points per rank" % (msm_log - (world.bit_length() - 1))}
        res["msm_g1"].append(row)
        log("[bench] sharded MSM 2^%d: %.3f ms on %d GPUs vs %.3f ms on one, identical=%s (%.1f s)" % (
            msm_log, t_msm, world, t_single, row["identical"], time.time() - t0))
    comm.close()
    res["identical"] = bool(res["proof"]["identical"] and all(r_["identical"] for r_ in res["ntt"] + res["msm_g1"]))
    return res


def run_sweep(args):
    """BASELINE.json configs[2..3] on one B200 with the CPU path beside every row: G1 / G2 MSM 2^16 .. 2^26 (G2 .. 2^24) and
    Fr NTT 2^16 .. 2^26, kernel-only with inputs resident in HBM (CUDA events, best of 5).  cpu_baseline per row
    (this is bench.py's cpu_baseline leg: the only place that may execute oracle/): CPU-B = the C port's Pippenger /
    iterative NTT on all host threads up to 2^22, CPU-A = its snarkjs-structured arithmetic (one double-and-add per
    point, recursive radix-2 FFT) on one thread up to 2^16 (MSM) / 2^20 (NTT).  Checks: every MSM result == (sum k_i s_i
    mod r) G with the sum (numpy) and the scalar multiplication (Python ints) on the host -- for the uniform, the
    rollup-like and every adversarial scalar set of SURVEY 8(d) config 3 (iii); every NTT on x_j = c g^j against the
    closed form at 8 random + first + last indices, plus the round trip."""
    import numpy as np
    import torch
    from oracle import cbind
    from simple_zk_rollups_b200 import _lib, prover
    L = _lib.lib()
    gp = prover.Groth16Prover(0)
    ctx = gp.ctx
    stream = torch.cuda.current_stream()
    _lib.check(L.zkr_ctx_set_stream(ctx, C.c_void_p(stream.cuda_stream)))
    cores = os.cpu_count() or 1
    imad_peak, modmul_peak, ms_mb = C.c_double(), C.c_double(), C.c_float()
    _lib.check(L.zkr_microbench(ctx, 0, 100000, C.byref(imad_peak), C.byref(ms_mb)))
    _lib.check(L.zkr_microbench(ctx, 2, 20000, C.byref(modmul_peak), C.byref(ms_mb)))
    res = {"what": "bench.py --sweep (one B200)", "imad_peak_per_s": imad_peak.value, "modmul_peak_per_s": modmul_peak.value,
           "host_threads": cores, "msm": [], "ntt": []}
    rng = np.random.default_rng(2026)

    def timeit(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return min(ts), float(np.median(ts))

    def w_model(n):
        return min(-(-255 // c) * 10.0 * n + 28.0 * (1 << (c - 1)) for c in range(4, 24))

    def wall(fn):
        t0 = time.time()
        fn()
        return time.time() - t0

    def host_g2_check(out, e):                     # G2 expectation: one fixed-base multiplication on the GPU (other kernel)
        if e % R_ORDER == 0:
            return out == bytes(128)               # the point at infinity is encoded as zeros
        esc = np.frombuffer(int(e).to_bytes(32, "little"), dtype=np.uint8).copy()
        exp_m = np.empty(128, dtype=np.uint8)
        _lib.check(L.zkr_synth_points(ctx, 2, _lib.buf_ptr(esc), 1, _lib.buf_ptr(exp_m)))
        rinv = pow(1 << 256, -1, Q_FIELD)
        exp = b"".join((int.from_bytes(exp_m[i:i + 32].tobytes(), "little") * rinv % Q_FIELD).to_bytes(32, "little")
                       for i in range(0, 128, 32))
        return exp == out

    for group, lo_log, hi_log in ((1, 16, args.sweep_max_log), (2, 16, min(24, args.sweep_max_log))):
        if "msm" not in args.sweep:
            break
        for lg in range(lo_log, hi_log + 1, 2):
            n = 1 << lg
            t0 = time.time()
            s64 = rng.integers(1, 1 << 63, size=n, dtype=np.uint64)
            sc_pts = np.zeros((n, 32), dtype=np.uint8)
            sc_pts[:, :8] = s64.view(np.uint8).reshape(n, 8)
            ab = 64 if group == 1 else 128
            pts = np.empty(n * ab, dtype=np.uint8)
            _lib.check(L.zkr_synth_points(ctx, group, _lib.buf_ptr(sc_pts), n, _lib.buf_ptr(pts)))
            bases = C.c_void_p()
            _lib.check(L.zkr_bases_load(ctx, group, _lib.buf_ptr(pts), n, 0, C.byref(bases)))
            cc, ww, nbytes = C.c_int(), C.c_int(), C.c_uint64()
            _lib.check(L.zkr_bases_info(bases, None, C.byref(cc), C.byref(ww), C.byref(nbytes)))
            t_load = time.time() - t0
            ssum = int((s64 & np.uint64(0xFFFFFFFF)).sum(dtype=np.uint64)) + (int((s64 >> np.uint64(32)).sum(dtype=np.uint64)) << 32)
            uni = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
            uni[:, 31] &= 0x1F
            roll = uni.copy()
            sel = rng.random(n) < 0.03
            roll[sel] = 0
            roll[sel, 0] = rng.integers(0, 2, size=int(sel.sum()), dtype=np.uint8)
            const = lambda k: np.tile(np.frombuffer(int(k).to_bytes(32, "little"), dtype=np.uint8), (n, 1))
            k_eq = 0x1234567890ABCDEF1234567890ABCDEF % R_ORDER
            alt = const(7)
            alt[1::2] = np.frombuffer(int(R_ORDER - 7).to_bytes(32, "little"), dtype=np.uint8)
            sets = [("uniform", uni, None), ("rollup_like", roll, None), ("all_zero", const(0), 0),
                    ("all_one", const(1), ssum % R_ORDER), ("all_rm1", const(R_ORDER - 1), (R_ORDER - 1) * ssum % R_ORDER),
                    ("all_equal", const(k_eq), k_eq * ssum % R_ORDER), ("alternating_k_rmk", alt, None)]
            mm = w_model(n) * (1 if group == 1 else 3)
            for name, arr, e in sets:
                if lg > 22 and name not in ("uniform", "rollup_like", "all_equal"):
                    continue                                    # host-side scalar sets of 2^24+ x 32 B: keep the run short
                k = np.ascontiguousarray(arr)
                if e is None:
                    e = dot_mod_r(k.reshape(-1), s64)
                d_k = torch.from_numpy(k.reshape(-1)).cuda()
                d_out = torch.zeros(256, dtype=torch.uint8, device="cuda")
                best, med = timeit(lambda: _lib.check(L.zkr_msm_dev(ctx, bases, C.c_void_p(d_k.data_ptr()), n, C.c_void_p(d_out.data_ptr()))))
                out = np.zeros(ab, dtype=np.uint8)
                _lib.check(L.zkr_msm(ctx, bases, C.c_void_p(d_k.data_ptr()), n, 1, _lib.buf_ptr(out)))
                ok = (out.tobytes() == host_g1_mul(e)) if group == 1 else host_g2_check(out.tobytes(), e)
                row = dict(group=group, log_n=lg, scalars=name, c=cc.value, windows=ww.value, ms_best=round(best, 4),
                           ms_median=round(med, 4), gpts_per_s=round(n / best / 1e6, 4), modmul_model=mm,
                           frac_of_modmul_peak=round(mm / (best * 1e-3) / modmul_peak.value, 4),
                           imad_frac_plain=round(mm * MODMUL_IMAD / (best * 1e-3) / imad_peak.value, 4),
                           table_gb=round(nbytes.value / 1e9, 3), load_s=round(t_load, 2), correct=bool(ok))
                if name == "uniform":
                    cpu = {}
                    if lg <= 22:
                        box = {}
                        tb = wall(lambda: box.update(r=cbind.msm(group, pts, k.reshape(-1), mode=1, threads=cores)))
                        same = box["r"] == out.tobytes()
                        cpu["cpu_b"] = dict(kind="port", algo="Pippenger, C restatement", cores=cores, seconds=round(tb, 3),
                                            gpts_per_s=round(n / tb / 1e9, 6), gpu_speedup=round(tb * 1e3 / best, 1), result_equal=same)
                    if lg <= 16:
                        ta = wall(lambda: box.update(r=cbind.msm(group, pts, k.reshape(-1), mode=0, threads=1)))
                        cpu["cpu_a"] = dict(kind="port", algo="snarkjs structure: one double-and-add per point", cores=1,
                                            seconds=round(ta, 3), gpts_per_s=round(n / ta / 1e9, 6), gpu_speedup=round(ta * 1e3 / best, 1),
                                            result_equal=box["r"] == out.tobytes())
                    row["cpu_baseline"] = cpu
                res["msm"].append(row)
                print(json.dumps(row), flush=True)
                del d_k
            L.zkr_bases_free(bases)
            del pts
    cval, gval = 0x1234567890ABCDEF1234567890ABCDEF0F1E2D3C4B5A6978 % R_ORDER, 0x0FEDCBA9876543210FEDCBA987654321 % R_ORDER
    cb = np.frombuffer(cval.to_bytes(32, "little"), dtype=np.uint8)
    gb = np.frombuffer(gval.to_bytes(32, "little"), dtype=np.uint8)
    import random
    for lg in range(16, (args.sweep_max_log if "ntt" in args.sweep else 0) + 1, 2):
        n = 1 << lg
        w = pow(5, (R_ORDER - 1) >> lg, R_ORDER)
        gsh = pow(5, (R_ORDER - 1) >> (lg + 1), R_ORDER)
        d = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        fill = lambda: _lib.check(L.zkr_fill_geometric(ctx, C.c_void_p(d.data_ptr()), n, _lib.buf_ptr(cb), _lib.buf_ptr(gb), 0, lg, 1, 0))
        val = lambda k: int.from_bytes(d[32 * k:32 * k + 32].cpu().numpy().tobytes(), "little")
        prng = random.Random(lg)
        probes = [0, n - 1] + [prng.randrange(n) for _ in range(8)]
        brev = lambda x: int(bin(x)[2:].zfill(lg)[::-1], 2)
        ok = True
        # forward (natural in, bit-reversed out): X[k] = c (g^N - 1) / (g w^k - 1)
        fill()
        _lib.check(L.zkr_ntt(ctx, C.c_void_p(d.data_ptr()), lg, 0 | 0x10, 1))
        top = cval * (pow(gval, n, R_ORDER) - 1) % R_ORDER
        for p_ in probes:
            ok = ok and val(p_) == top * pow((gval * pow(w, brev(p_), R_ORDER) - 1) % R_ORDER, -1, R_ORDER) % R_ORDER
        # coset forward: X[k] = x(gsh w^k) = c ((g gsh)^N - 1) / (g gsh w^k - 1)
        fill()
        _lib.check(L.zkr_ntt(ctx, C.c_void_p(d.data_ptr()), lg, 2 | 0x10, 1))
        g2 = gval * gsh % R_ORDER
        top2 = cval * (pow(g2, n, R_ORDER) - 1) % R_ORDER
        for p_ in probes[:5]:
            ok = ok and val(p_) == top2 * pow((g2 * pow(w, brev(p_), R_ORDER) - 1) % R_ORDER, -1, R_ORDER) % R_ORDER
        # round trip: DIT^-1(DIF(x)) == x
        fill()
        _lib.check(L.zkr_ntt(ctx, C.c_void_p(d.data_ptr()), lg, 0 | 0x10, 1))
        _lib.check(L.zkr_ntt(ctx, C.c_void_p(d.data_ptr()), lg, 1 | 0x20, 1))
        ref = torch.empty_like(d)
        _lib.check(L.zkr_fill_geometric(ctx, C.c_void_p(ref.data_ptr()), n, _lib.buf_ptr(cb), _lib.buf_ptr(gb), 0, lg, 1, 0))
        torch.cuda.synchronize()
        ok = ok and bool(torch.equal(ref, d))
        del ref
        cpu = {}
        if lg <= 22:
            x = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
            x[:, 31] &= 0x1F
            xb = np.ascontiguousarray(x).reshape(-1)
            tb = wall(lambda: cbind.ntt(xb.copy(), lg, False, False, 1, cores))
            cpu["cpu_b"] = dict(kind="port", algo="iterative radix-2, C restatement", cores=cores, seconds=round(tb, 4),
                                gb_per_s=round(64.0 * n / tb / 1e9, 3))
            if lg <= 20:
                ta = wall(lambda: cbind.ntt(xb.copy(), lg, False, False, 0, 1))
                cpu["cpu_a"] = dict(kind="port", algo="snarkjs polfield structure: recursive radix-2", cores=1, seconds=round(ta, 4),
                                    gb_per_s=round(64.0 * n / ta / 1e9, 3))
        for name, mode in (("forward_dif", 0 | 0x10), ("inverse_dit", 1 | 0x20), ("coset_forward_dif", 2 | 0x10)):
            best, med = timeit(lambda: _lib.check(L.zkr_ntt(ctx, C.c_void_p(d.data_ptr()), lg, mode, 1)))
            mm = (n // 2) * lg
            row = dict(log_n=lg, op=name, ms_best=round(best, 4), ms_median=round(med, 4), gb_per_s=round(64.0 * n / (best * 1e-3) / 1e9, 1),
                       butterfly_modmul_frac_of_peak=round(mm / (best * 1e-3) / modmul_peak.value, 4),
                       imad_frac_plain=round(mm * MODMUL_IMAD / (best * 1e-3) / imad_peak.value, 4), correct=bool(ok))
            if name == "forward_dif":
                row["cpu_baseline"] = cpu
                for kk in cpu.values():
                    kk["gpu_speedup"] = round(kk["seconds"] * 1e3 / best, 1)
            res["ntt"].append(row)
            print(json.dumps(row), flush=True)
        del d
    gp.close()
    if args.sweep_out:
        os.makedirs(os.path.dirname(args.sweep_out) or ".", exist_ok=True)
        json.dump(res, open(args.sweep_out, "w"), indent=1)


def _lib_check(rc):
    from simple_zk_rollups_b200 import _lib
    _lib.check(rc)


def _buf_ptr(b):
    from simple_zk_rollups_b200 import _lib
    return _lib.buf_ptr(b)


def _Stats():
    from simple_zk_rollups_b200 import _lib
    return _lib.Stats()


def cpu_baseline(pk_bin, wbytes, rs, gpu_proof, args):
    """oracle/c (kind 'port') on all host cores; one full proof of the same workload, checked against the GPU's."""
    from oracle import cbind
    cores = os.cpu_count() or 1
    t0 = time.time()
    got = cbind.prove(pk_bin, wbytes, rs[0], rs[1], mode=1, threads=cores)
    dt = time.time() - t0
    ok = got == gpu_proof
    log("[bench] cpu_baseline: %.2f s per proof on %d threads; proof %s the GPU's" % (dt, cores, "==" if ok else "!="))
    return {"value": round(1.0 / dt, 5), "unit": "proofs/s", "cores": cores, "kind": "port",
            "sample": "1 full proof of the same workload (same key, witness, r, s); Pippenger + iterative NTT, "
                      "websnark calcH structure; proof bytes %s the GPU proof" % ("equal" if ok else "DIFFER FROM"),
            "seconds_per_proof": round(dt, 3), "matches_gpu_proof": ok}


def run_reference(args):
    """Reference arm: the CPU port of the reference's algorithm, all host threads, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    from oracle import cbind
    from simple_zk_rollups_b200 import synth
    cbind.build()
    cores = os.cpu_count() or 1
    r1, w = make_workload(args.shape, seed=11)
    wbytes = synth.witness_bytes(w)
    # The proving key is workload data, not code under test, and only the GPU setup can make one at this size (the
    # Python oracle's setup is per-point big-int work).  It is made by a CHILD process (bench.py --make-key), so this
    # process -- the one that is timed -- never maps libzkr.so or touches the GPU; a key file left by an earlier run
    # of the same shape is reused.
    import tempfile
    key_path = os.path.join(tempfile.gettempdir(), "zkr_ref_key_%s.bin" % args.shape)     # hundreds of MB: not in the repo tree
    if not os.path.exists(key_path):
        env = dict(os.environ)
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--make-key", key_path, "--shape", args.shape],
                           env=env, capture_output=True, text=True)
        if p.returncode != 0:
            log("[bench] key generation child failed: %s" % (p.stderr.strip().splitlines() or ["?"])[-1])
    if not os.path.exists(key_path):
        print(json.dumps({"impl": "reference", "unavailable": "no proving key for the workload (the synthetic setup needs a GPU)"}))
        return
    pk_bin = np.fromfile(key_path, dtype=np.uint8)
    rs = RS
    mode = args.ref_mode
    if args.ref_threads:
        cores = args.ref_threads
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.time()
        proof = cbind.prove(pk_bin, wbytes, rs[0], rs[1], mode=mode, threads=cores)
        dt = time.time() - t0
        if i >= args.warmup:
            times.append(dt)
        log("[bench] reference step %d: %.2f s" % (i, dt))
    if args.dump_outputs:
        dump_proof(args.dump_outputs, "proof", proof)
    total = sum(times)
    val = len(times) / total
    n = r1.nVars
    bits, m = r1.domain()
    print(json.dumps({
        "impl": "reference", "metric": "groth16_proofs_per_s", "value": round(val, 5), "unit": "proofs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / len(times), 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (4x64-bit-limb Montgomery)",
        "data": "synthetic",
        "config": {"workload": workload_string(args.shape, r1, n, bits),
                   "key_resident_in_hbm": False,
                   "baseline_config": BASELINE_CONFIG.get(args.shape, "BASELINE.json configs[1] shape family")},
        "cpu_baseline": {"value": round(val, 5), "unit": "proofs/s", "cores": cores, "kind": "port",
                         "sample": "every step is 1 full proof of the workload (C restatement of websnark groth16GenProof: "
                                   + ("Pippenger multiexp + iterative NTT" if mode == 1 else
                                      "snarkjs arithmetic structure: one double-and-add multiplication per point, recursive radix-2 FFT")
                                   + ", %d host thread(s))" % cores},
        "e2e": {"value": round(val, 5), "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def make_key(args):
    """Child of the reference arm: synthetic proving key of the workload -> file (GPU setup; workload data only)."""
    from simple_zk_rollups_b200 import keygen, prover
    r1, _ = make_workload(args.shape, seed=11)
    gp = prover.Groth16Prover(0)
    pk_bin, _ = keygen.synth_setup(gp.ctx, r1, TOXIC)
    gp.close()
    tmp = args.make_key + ".tmp%d" % os.getpid()
    pk_bin.tofile(tmp)
    os.replace(tmp, args.make_key)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="tx_2p20", help="withdraw | tx | tx_2p20 | tx_2p22 (simple_zk_rollups_b200.synth.SHAPES)")
    ap.add_argument("--ref-mode", type=int, default=1, choices=[0, 1],
                    help="--impl reference: 1 = Pippenger + iterative NTT (default), 0 = snarkjs arithmetic structure (SURVEY 8(d) CPU-A)")
    ap.add_argument("--ref-threads", type=int, default=0, help="--impl reference: host threads (default: all)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs under ncu)")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the sharded proof / NTT / MSM block")
    ap.add_argument("--no-gpu-witness", action="store_true", help="skip the witness-on-GPU block")
    ap.add_argument("--in-flight", type=int, default=2, help="contexts / key replicas per GPU in the e2e leg (default 2)")
    ap.add_argument("--no-two-in-flight", action="store_true", help="skip the e2e leg with two contexts / key replicas per GPU")
    ap.add_argument("--no-batch-2p22", action="store_true", help="skip the BASELINE configs[4] batch block")
    ap.add_argument("--sharded-ntt-logs", default="24,26")
    ap.add_argument("--sharded-msm-log", default="24", help="comma list of log2 sizes of the sharded G1 MSM")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the proof of the last timed step as DIR/proof.npy (float64, 8 coordinates x 32 bytes)")
    ap.add_argument("--make-key", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--sweep", default="", help="msm,ntt: BASELINE configs[2..3] sweeps on one GPU with CPU baselines beside every row")
    ap.add_argument("--sweep-max-log", type=int, default=26)
    ap.add_argument("--sweep-out", default=None)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.make_key:
        make_key(args)
        return
    if args.sweep:
        run_sweep(args)
        return
    if args.warmup < 3 and args.impl == "ours":
        log("[bench] note: timing rules ask for >= 3 warm-up steps")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
