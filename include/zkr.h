/* zkr.h -- C ABI of the B200-native BN254 Groth16 prover for simple-zk-rollups.
 *
 * This is the drop-in boundary for the proof-generation hot path of
 * kendricktan/simple-zk-rollups.  Each entry point replaces one call the reference makes
 * into its (un-vendored) websnark / snarkjs dependencies; citations are relative to the
 * reference tree:
 *
 *   zkr_ctx_create        <-> buildBn128()                    operator/src/snarks/common.ts:23
 *   zkr_pkey_load_bin     <-> consumes binarifyProvingKey()   operator/src/utils/binarify.ts:50-207
 *                             output; done ONCE per circuit instead of per proof (common.ts:28)
 *   zkr_prove             <-> wasmBn128.groth16GenProof(witnessBin, provingKeyBin)
 *                                                             operator/src/snarks/common.ts:29
 *                             witnessBin = binarifyWitness()  operator/src/utils/binarify.ts:10-48
 *   zkr_prove_batch       <-> many independent genTxVerifierProof calls (tx.ts:6-10), one per GPU
 *   zkr_msm_* / zkr_ntt   <-> websnark g1_multiexp / g2_multiexp / fft_* (inside groth16GenProof);
 *                             exported for the standalone sweeps of BASELINE.json configs[2..3]
 *   zkr_synth_setup       <-> `snarkjs setup --protocol groth`  prover/package.json:34,37
 *                             (synthetic keys only: toxic waste is an input)
 *   zkr_setup_from_powers <-> the same, as a deployable key: from public powers of tau, then
 *   zkr_setup_contribute      phase-2 delta contributions that anyone can check
 *                             (zkr_setup_verify_contribution)
 *
 * Conventions
 *   - All multi-byte integers little-endian.  Field elements are 32 bytes = 8 x u32 limbs,
 *     least-significant first (binarify.ts:68-76).
 *   - "Fq-M"/"Fr-M" = Montgomery form, radix 2^256 (binarify.ts:78-90); "std" = plain value.
 *   - Every function returns 0 on success or a negative ZKR_E_* code; zkr_last_error()
 *     returns a thread-local message.  There is NO CPU fallback: without a usable sm_100
 *     device every compute entry point fails with ZKR_E_NO_DEVICE / ZKR_E_CUDA.
 *   - Input buffers are borrowed for the duration of the call; outputs are caller-allocated.
 *     zkr_ctx / zkr_pkey / zkr_bases are opaque handles owned by the library until freed.
 *   - Calls on one zkr_ctx are serialised by the caller (one ctx per thread / per GPU).
 */
#ifndef ZKR_H
#define ZKR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZKR_OK 0
#define ZKR_E_INVALID (-1)        /* bad argument */
#define ZKR_E_BADKEY (-2)         /* proving-key buffer fails structural validation */
#define ZKR_E_WITNESS_RANGE (-3)  /* a witness / scalar value is >= r, or witness[0] != 1 */
#define ZKR_E_CUDA (-4)           /* CUDA runtime error (message has the detail) */
#define ZKR_E_NO_DEVICE (-5)      /* no CUDA device / not an sm_100 part */
#define ZKR_E_NOMEM (-6)
#define ZKR_E_NCCL (-7)
#define ZKR_E_UNSUPPORTED (-8)

#define ZKR_PROOF_BYTES 256

typedef struct zkr_ctx zkr_ctx;
typedef struct zkr_pkey zkr_pkey;
typedef struct zkr_bases zkr_bases;

/* Per-stage device times of the last zkr_prove on this ctx, milliseconds (CUDA events). */
typedef struct zkr_stats {
    float total_ms;      /* first kernel launch .. proof bytes on host */
    float h2d_ms;        /* witness upload */
    float lc_ms;         /* sparse A_T, B_T */
    float ntt_ms;        /* H pipeline (6 NTTs + pointwise) */
    float msm_a_ms, msm_b1_ms, msm_b2_ms, msm_c_ms, msm_h_ms;
    float assemble_ms;
    uint64_t kernel_launches; /* kernels of this library launched by the call */
} zkr_stats;

const char* zkr_strerror(int code);
const char* zkr_last_error(void);
/* library / build identification, e.g. "zkr 0.1 sm_100a" */
const char* zkr_version(void);

/* ---- context ------------------------------------------------------------------------ */
int zkr_ctx_create(int device, zkr_ctx** out);
void zkr_ctx_destroy(zkr_ctx* ctx);
/* Order all subsequent work of this ctx after / before `stream` (a cudaStream_t, may be
 * NULL = legacy default stream): the library forks its internal streams off it and joins
 * them back, so CUDA events recorded on `stream` bracket the library's kernels. */
int zkr_ctx_set_stream(zkr_ctx* ctx, void* stream);
int zkr_ctx_synchronize(zkr_ctx* ctx);
/* number of this library's kernels launched through ctx since creation */
uint64_t zkr_ctx_kernel_launches(const zkr_ctx* ctx);

/* Per-kernel device timing (CUDA events on the launching stream) for roofline reporting.
 * id: 0 = G1 bucket accumulation (k_accum_affine<Fq>), 1 = G2 bucket accumulation, 2 = NTT pass (local),
 *     3 = the NTT pass of a sharded transform whose write-back is the all-to-all (remote stores).
 * units: work summed over the recorded launches -- mixed additions for ids 0/1, elements for ids 2/3. */
int zkr_ctx_set_profile(zkr_ctx* ctx, int on);
/* on != 0: zkr_prove runs its stages back to back on the ctx stream instead of forking five streams
 * (isolated per-kernel timings; the default overlaps the MSMs and the H pipeline). */
int zkr_ctx_set_serial(zkr_ctx* ctx, int on);
int zkr_ctx_profile_read(zkr_ctx* ctx, int id, double* total_ms, int* launches, double* units);

/* plain device-memory helpers on ctx's GPU (stream-ordered on the ctx stream; download synchronises).
 * They let a host language without a CUDA binding stage "already resident" inputs. */
int zkr_dev_malloc(zkr_ctx* ctx, size_t bytes, void** d_out);
int zkr_dev_free(zkr_ctx* ctx, void* d_ptr);
int zkr_dev_upload(zkr_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
int zkr_dev_download(zkr_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);

/* ---- proving key -------------------------------------------------------------------- */
/* Parse the websnark binary proving key (binarify.ts:152-202 layout, SURVEY.md A.1), convert
 * polsA/polsB to row-major CSR, compact + window-precompute the five base sets, keep all of it
 * resident in HBM.  buf may be host memory; it is not referenced after return. */
int zkr_pkey_load_bin(zkr_ctx* ctx, const void* buf, size_t len, zkr_pkey** out);
void zkr_pkey_free(zkr_pkey* pk);
int zkr_pkey_info(const zkr_pkey* pk, uint32_t* n_vars, uint32_t* n_public, uint32_t* domain_size,
                  uint64_t* device_bytes);

/* ---- key / witness ingestion from the snarkjs JSON text (SURVEY.md 8(f) rank 1) ------------ */
/* binarifyProvingKey (operator/src/utils/binarify.ts:50-207) applied to the TEXT of a snarkjs
 * `--protocol groth` proving key (proving_key.json, fields per SURVEY.md A.3): one streaming pass,
 * output byte-identical to the reference's ArrayBuffer.  Values may be decimal strings
 * (stringifyBigInts) or bare JSON integers; key order is free; polsC and unknown fields are
 * skipped.  *out_buf is allocated by the library: release it with zkr_buf_free.  Host-only
 * (no device needed).  Errors: ZKR_E_BADKEY (message names the byte offset), ZKR_E_UNSUPPORTED
 * if the layout would exceed the format's 32-bit offsets, ZKR_E_NOMEM. */
int zkr_pkey_json_to_bin(const char* json, size_t len, void** out_buf, size_t* out_len);
/* binarifyWitness (binarify.ts:10-48) applied to the text of a witness.json (array of decimal
 * strings / integers): n x 32 B little-endian, std form, values written as is. */
int zkr_witness_json_to_bin(const char* json, size_t len, void** out_buf, size_t* out_len);
void zkr_buf_free(void* buf);
/* zkr_pkey_json_to_bin + zkr_pkey_load_bin: what replaces
 * `binarifyProvingKey(provingKey)` at operator/src/snarks/common.ts:28, once per circuit. */
int zkr_pkey_load_json(zkr_ctx* ctx, const char* json, size_t len, zkr_pkey** out);

/* ---- prove -------------------------------------------------------------------------- */
/* witness: n_signals x 32 B std form (binarifyWitness layout), HOST memory.
 * r32 / s32: blinding scalars, 32 B std form < r.  NULL = the library draws the scalar uniformly from
 *   [0, r) with the OS CSPRNG (getrandom), as websnark's groth16GenProof does internally: a caller who
 *   passes nothing gets a zero-knowledge proof.  The snarkjs debug mode (r = s = 0: deterministic, NOT
 *   zero-knowledge) and fixed-(r, s) parity runs pass explicit buffers.  The sharded prove needs the same
 *   (r, s) on every rank and therefore rejects NULL.
 * out_proof: 256 B = pi_a (x|y) | pi_b (x.c0|x.c1|y.c0|y.c1) | pi_c (x|y), std form, affine,
 *   i.e. exactly the integers websnark prints as decimal strings (z omitted: "1" / ["1","0"]).
 *   A point at infinity is encoded as all-zero coordinates. */
int zkr_prove(zkr_ctx* ctx, const zkr_pkey* pk, const void* witness, size_t n_signals,
              const void* r32, const void* s32, void* out_proof, zkr_stats* stats);
/* Same with the witness already resident in device memory of ctx's GPU (d_witness) and the
 * proof written to device memory (d_out_proof, 256 B); asynchronous w.r.t. the host, ordered
 * on the ctx stream (zkr_ctx_set_stream).  Being asynchronous it cannot return
 * ZKR_E_WITNESS_RANGE: invalid inputs (a value >= r, witness[0] != 1) give a meaningless proof and
 * set device-side flags that stay set until zkr_prove_check reads them.  zkr_prove and
 * zkr_prove_batch start from clean flags and report on their own inputs only. */
int zkr_prove_dev(zkr_ctx* ctx, const zkr_pkey* pk, const void* d_witness, size_t n_signals,
                  const void* r32, const void* s32, void* d_out_proof);
/* Synchronise the ctx stream, then report and clear the input-validity flags of every zkr_prove_dev
 * on `pk` since the last check: ZKR_OK or ZKR_E_WITNESS_RANGE. */
int zkr_prove_check(zkr_ctx* ctx, const zkr_pkey* pk);
/* n_proofs independent proofs over n_ctx contexts (one per GPU; pks[i] is the same key loaded on
 * ctxs[i]'s device), scheduled round-robin, one in flight per GPU.  witnesses: n_proofs buffers. */
int zkr_prove_batch(zkr_ctx* const* ctxs, const zkr_pkey* const* pks, int n_ctx,
                    const void* const* witnesses, size_t n_signals, int n_proofs,
                    const void* rs32 /* n_proofs x 64 B (r|s), or NULL = fresh CSPRNG pairs */, void* out_proofs);

/* ---- witness generation for forward-solvable constraint systems (SURVEY.md 8(f) rank 4) ---------
 * Stands where the reference calls circom's generated calculator, circuit.calculateWitness(inputs)
 * (operator/src/snarks/common.ts:12-17), for circuits whose constraints each introduce at most one new
 * signal -- the one with the largest index -- and only in C:  new = ((A.w)(B.w) - C'.w) / c_new.  MiMC /
 * Feistel rounds (prover/circuits/hasher.circom:8), products and linear combinations are of this form;
 * signals no constraint defines that way (circuit inputs, bits under b (b - 1) = 0, circom `<--` hints)
 * are GIVEN by the caller.  zkr_wprog_build analyses the R1CS once per circuit (r1cs: the circuit's own
 * constraints, WITHOUT the input-consistency rows a snarkjs setup adds to polsA; zkr_r1cs_csc is declared
 * below); ZKR_E_UNSUPPORTED if a row uses a signal that only a later row defines.
 * zkr_wprog_given lists the signals the caller must supply (ascending; signal 0, the constant 1, is one
 * of them).  zkr_witness_solve takes their values (n_given x 32 B std form, HOST memory, that order) and
 * leaves the complete witness in DEVICE memory (d_witness: n_vars x 32 B std form), ready for
 * zkr_prove_dev: one kernel launch per level of the dependency graph, no host round trip.
 * Errors: ZKR_E_WITNESS_RANGE if a given value is >= r. */
typedef struct zkr_wprog zkr_wprog;
struct zkr_r1cs_csc;
int zkr_wprog_build(zkr_ctx* ctx, const struct zkr_r1cs_csc* r1cs, zkr_wprog** out);
void zkr_wprog_free(zkr_wprog* wp);
int zkr_wprog_info(const zkr_wprog* wp, uint32_t* n_vars, uint32_t* n_given, uint32_t* n_solved, uint32_t* n_levels);
int zkr_wprog_given(const zkr_wprog* wp, uint32_t* out_signals /* n_given */);
int zkr_witness_solve(zkr_ctx* ctx, const zkr_wprog* wp, const void* given_values, void* d_witness);

/* ---- verify (SURVEY.md 8(f) rank 2) -------------------------------------------------- */
/* Replaces snarkjs groth.isValid(verifyingKey, proof, publicSignals) at
 * operator/src/snarks/common.ts:30-34 with the on-chain predicate of
 * contracts/contracts/TxVerifier.sol:258-276:
 *   vk_x = IC[0] + sum input[i] IC[i+1];  e(-A,B) e(alfa1,beta2) e(vk_x,gamma2) e(C,delta2) == 1.
 * The l-term MSM for vk_x runs on ctx's GPU over IC tables kept resident per verifying key; the
 * 4-pairing product runs on the calling host thread (O(1) work, ~2 ms).
 * zkr_vkey_load_json: text of a snarkjs verification_key.json (SURVEY.md A.3).
 * zkr_vkey_load_bin:  alfa1|beta1|delta1 (64 B each) | beta2|gamma2|delta2 (128 B each) | IC[0..l]
 *                     (64 B each), Fq-M -- the vk block zkr_synth_setup emits.
 * Both validate every point (on curve; G2 in the order-r subgroup) -> ZKR_E_BADKEY otherwise. */
typedef struct zkr_vkey zkr_vkey;
int zkr_vkey_load_json(zkr_ctx* ctx, const char* json, size_t len, zkr_vkey** out);
int zkr_vkey_load_bin(zkr_ctx* ctx, const void* buf, size_t len, zkr_vkey** out);
void zkr_vkey_free(zkr_vkey* vk);
int zkr_vkey_info(const zkr_vkey* vk, uint32_t* n_public);
/* proof: 256 B in zkr_prove's output encoding.  public_signals: n_public x 32 B std form, HOST memory.
 * *valid = 1 iff the predicate holds; malformed proof points (coordinate >= q, off curve, B outside the
 * subgroup) give *valid = 0.  Errors mirror the contract's reverts: n_public != nPublic of the key ->
 * ZKR_E_INVALID ("verifier-bad-input", TxVerifier.sol:261); a signal >= r -> ZKR_E_WITNESS_RANGE
 * ("verifier-gte-snark-scalar-field", :265). */
int zkr_verify(zkr_ctx* ctx, const zkr_vkey* vk, const void* proof, const void* public_signals,
               size_t n_public, int* valid);
/* prod_i e(P_i, Q_i) == 1 for n <= 8 pairs; g1_points n x 64 B, g2_points n x 128 B (x.c0|x.c1|y.c0|y.c1),
 * std form affine, all-zero = infinity: the alt_bn128 pairing-check TxVerifier.sol:91-116 calls.
 * Host-only.  Invalid inputs (>= q, off curve, G2 outside the subgroup) -> ZKR_E_INVALID, like the
 * precompile failing. */
int zkr_pairing_check(const void* g1_points, const void* g2_points, size_t n, int* is_one);

/* ---- standalone MSM ----------------------------------------------------------------- */
/* group: 1 = G1 (64 B affine Fq-M points), 2 = G2 (128 B, x.c0|x.c1|y.c0|y.c1).
 * points: host memory, n of them; x == 0 marks infinity (skipped).  Builds the windowed
 * precompute table in HBM (window_bits = 0 -> chosen from n). */
int zkr_bases_load(zkr_ctx* ctx, int group, const void* points, size_t n, int window_bits,
                   zkr_bases** out);
void zkr_bases_free(zkr_bases* b);
int zkr_bases_info(const zkr_bases* b, uint64_t* n_points, int* window_bits, int* n_windows,
                   uint64_t* device_bytes);
/* sum_i scalars[i] * points[i]; scalars n x 32 B std form (< r), host memory if scalars_on_device
 * == 0 else device memory.  out: affine std form, 64 B (G1) or 128 B (G2), host memory. */
int zkr_msm(zkr_ctx* ctx, const zkr_bases* b, const void* scalars, size_t n, int scalars_on_device,
            void* out_affine);
/* device-resident, asynchronous variant: result stays on the device as an XYZZ point
 * (4 coordinates Fq-M / Fq2-M: 128 B for G1, 256 B for G2). */
int zkr_msm_dev(zkr_ctx* ctx, const zkr_bases* b, const void* d_scalars, size_t n, void* d_out_xyzz);

/* ---- standalone NTT over Fr ----------------------------------------------------------- */
#define ZKR_NTT_FORWARD 0       /* evaluations on <omega_n>, natural order in and out          */
#define ZKR_NTT_INVERSE 1       /* coefficients (includes the 1/n scaling)                      */
#define ZKR_NTT_COSET_FORWARD 2 /* evaluations on g<omega_n>, g = omega_2n                      */
#define ZKR_NTT_COSET_INVERSE 3
/* OR-able order flags: skip the bit-reversal pass on one side.  BITREV_OUT: natural in, result left
 * in bit-reversed order (pure DIF).  BITREV_IN: input given in bit-reversed order, natural out (pure
 * DIT).  The prover chains DIF^-1 -> DIT -> DIF^-1 and never runs a bit-reversal pass. */
#define ZKR_NTT_BITREV_OUT 0x10
#define ZKR_NTT_BITREV_IN 0x20
/* data: 2^log_n x 32 B Fr std form, transformed in place; on_device selects host / device memory.
 * omega_n = 5^((r-1)/n) (snarkjs PolField convention). */
int zkr_ntt(zkr_ctx* ctx, void* data, int log_n, int mode, int on_device);
/* The fused H pipeline of the prover (SURVEY.md B.4 method iv): a_t, b_t = A_T, B_T evaluations
 * (2^log_m x 32 B std form, device memory, clobbered); h_out receives h_0..h_{m-1} std form in
 * BIT-REVERSED order when bitrev_out != 0 (what the prover feeds to the hExps MSM) or natural order. */
int zkr_h_from_evals_dev(zkr_ctx* ctx, void* d_a_t, void* d_b_t, int log_m, void* d_h_out, int bitrev_out);
/* Workload generator for the NTT sweeps (BASELINE.json configs[3]): d_out[p] = c * g^j(p), std form, device
 * memory; c32, g32: 32 B std form, host.  world == 1: j(p) = start + p.  world = 2, 4, 8: d_out is `rank`'s
 * COLS slab (n_local = 2^log_n / world elements) of a zkr_ntt_sharded transform of 2^log_n elements, j(p)
 * the element's index in the whole vector (start ignored).  A dense vector whose transform the host can
 * check in closed form at any size: X[k] = sum_j c g^j w^(jk) = c (g^N - 1) / (g w^k - 1).
 * Asynchronous, ordered on the ctx stream. */
int zkr_fill_geometric(zkr_ctx* ctx, void* d_out, size_t n_local, const void* c32, const void* g32,
                       uint64_t start, int log_n, int world, int rank);

/* ---- multi-GPU: peer-memory communicator, sharded MSM, sharded four-step NTT ----------------
 * One zkr_comm per rank (GPU).  Each rank owns a device slab (flags | gather slots | two exchange
 * buffers of max_elems_per_rank Fr elements) that every peer maps, so kernels store directly into
 * peers' HBM over NVLink; there is no NCCL on the data path.  Wiring, across processes:
 *     zkr_comm_create -> zkr_comm_export (64 B handle) -> exchange the handles by any means
 *     (torch.distributed / MPI / a file) -> zkr_comm_connect(all handles, rank order);
 * inside one process (one ctx per GPU): zkr_comm_connect_local.  world = 1, 2, 4 or 8.
 * Replaces the web-worker fan-out of websnark's multiexp / fft inside groth16GenProof
 * (operator/src/snarks/common.ts:29) by a fan-out over the GPUs of one NVSwitch box. */
typedef struct zkr_comm zkr_comm;
#define ZKR_IPC_HANDLE_BYTES 64
int zkr_comm_create(zkr_ctx* ctx, int rank, int world, size_t max_elems_per_rank, zkr_comm** out);
int zkr_comm_export(const zkr_comm* c, void* handle64);
int zkr_comm_connect(zkr_comm* c, const void* handles /* world x 64 B, rank order */);
int zkr_comm_connect_local(zkr_comm* const* comms, int world);
/* device-side flag barrier across the ranks, ordered on the ctx stream (bounded spin: a missing peer
 * turns into ZKR_E_NCCL at the next zkr_comm_check / synchronising call, not a hang).  Every collective
 * entry point validates its arguments on the host BEFORE it launches a barrier, so a rank that returns
 * ZKR_E_INVALID has not half-entered a collective; if a barrier does time out (a peer died or bailed out
 * on a CUDA error) the ranks' barrier epochs may differ, the communicator is marked dead -- every later
 * call on it returns ZKR_E_NCCL -- and it must be destroyed and re-created on every rank. */
int zkr_comm_barrier(zkr_comm* c);
int zkr_comm_check(zkr_comm* c);
/* device pointer of this rank's exchange buffer 0 / 1 */
void* zkr_comm_buffer(zkr_comm* c, int which);
int zkr_comm_info(const zkr_comm* c, int* rank, int* world, uint64_t* elems_per_buffer);
void zkr_comm_destroy(zkr_comm* c);

/* MSM sharded by point range: `b` holds THIS rank's contiguous slice of the points (zkr_bases_load on
 * the slice), scalars the matching slice.  Each rank reduces its slice to one XYZZ point, stores it into
 * every peer's gather slot, and all ranks add the `world` partials: out_affine (as zkr_msm) is the
 * full sum on every rank. */
int zkr_msm_sharded(zkr_comm* c, const zkr_bases* b, const void* scalars, size_t n_local,
                    int scalars_on_device, void* out_affine);

/* One proof over `world` GPUs (latency split; SURVEY.md 8(e): "GPU0: sparse_lc + H + MSM_H; others: MSM_A, MSM_B1,
 * MSM_B2, MSM_C; combine 5 points" -- websnark fans the same calls out to web workers inside groth16GenProof,
 * operator/src/snarks/common.ts:29).  Every rank receives the full witness.  The first g_h ranks (the H group:
 * 1 of 2, 2 of 4, 4 of 8) compute A_T/B_T and h and run 1/g_h of the hExps MSM each (the H pipeline does not shard at
 * rollup sizes, so it is kept off the other ranks instead of being replicated on all of them); the four witness
 * MSMs (A, B1, B2, C; blinding bases included) are split by contiguous point range with weights that give every
 * rank the same modelled work (csrc/prover.cu shard_plan).  zkr_pkey_load_bin_sharded keeps only this rank's
 * ranges resident.  Each rank blinds its own partial A / B1 (scalar multiplication is linear), stores its seven
 * partial sums into every peer's gather slot, adds the `world` partials and assembles the proof.  All ranks return
 * the same 256 bytes, identical to zkr_prove on one GPU.  Same arguments and error behaviour as zkr_prove, except that
 * r32 / s32 are required (all ranks must use the same pair).
 * zkr_shard_ranges reports the split (no GPU needed): out6 = {ab_lo, ab_hi, c_lo, c_hi, h_lo, h_hi}, ranges of rank
 * over the n_vars + 2 points of A'/B1'/B2', the n_vars - n_public - 1 + 1 points of C', and the domain_size
 * coefficients of h (bit-reversed order; empty outside the H group). */
int zkr_shard_ranges(int world, int rank, uint64_t n_vars, uint64_t n_public, uint64_t domain_size, uint64_t* out6);
int zkr_pkey_load_bin_sharded(zkr_ctx* ctx, const void* buf, size_t len, int rank, int world, zkr_pkey** out);
int zkr_prove_sharded(zkr_comm* c, const zkr_pkey* pk, const void* witness, size_t n_signals,
                      const void* r32, const void* s32, void* out_proof, zkr_stats* stats);

/* Four-step NTT of 2^log_n elements sharded over the ranks, one all-to-all, fused into the pass that
 * precedes it (remote stores).  View the index as (row i, column j), i < 2^k0, j < 2^s0, k0 =
 * zkr_ntt_sharded_rows_log(log_n, world), s0 = log_n - k0, C = 2^s0:
 *   COLS slab of rank p: all rows, columns [p C/world, (p+1) C/world): local[i * C/world + jl] = x[i C + p C/world + jl]
 *   ROWS slab of rank q: the contiguous slice [q N/world, (q+1) N/world)
 * mode = ZKR_NTT_{FORWARD,INVERSE,COSET_FORWARD,COSET_INVERSE} | exactly one of
 *   ZKR_NTT_BITREV_OUT: input natural order in COLS slabs  -> output bit-reversed order in ROWS slabs
 *   ZKR_NTT_BITREV_IN : input bit-reversed order in ROWS slabs -> output natural order in COLS slabs
 * so transforms chain (DIF^-1 -> DIT -> DIF^-1, as the H pipeline does) with no extra exchange.
 * Input: this rank's slab in exchange buffer src_buf; output: exchange buffer 1 - src_buf.
 * Asynchronous, ordered on the ctx stream. */
int zkr_ntt_sharded_rows_log(int log_n, int world);
int zkr_ntt_sharded(zkr_comm* c, int log_n, int mode, int src_buf);

/* ---- synthetic trusted setup (test / benchmark keys only) ------------------------------ */
/* R1CS in CSC-by-signal form with coefficients taken from a pool:
 *   ptr_X[n_vars+1], row_X[nnz], cid_X[nnz] (u32), pool: n_pool x 32 B std form.
 * polsA must already contain the input-consistency rows (snarkjs setup_groth.js).
 * toxic: 5 x 32 B std form (tau, alpha, beta, gamma, delta).
 * Outputs (host buffers) are the POINT SECTIONS of the websnark binary proving key, encoded exactly
 * as binarifyProvingKey writes them (affine Fq-M, infinity = (0, R mod q)): out_a / out_b1 (64 n),
 * out_b2 (128 n), out_c (64 (n - n_public - 1)), out_h (64 domain_size); and out_vk =
 * alfa1 (64) | beta1 (64) | delta1 (64) | beta2 (128) | gamma2 (128) | delta2 (128) | IC[n_public+1] (64 each),
 * same encoding.  The host assembles header + pols sections around them (simple_zk_rollups_b200/keygen.py). */
typedef struct zkr_r1cs_csc {
    uint32_t n_vars, n_public, n_constraints, domain_size, n_pool;
    const uint32_t *ptr_a, *row_a, *cid_a;
    const uint32_t *ptr_b, *row_b, *cid_b;
    const uint32_t *ptr_c, *row_c, *cid_c;
    const void* pool;
} zkr_r1cs_csc;
int zkr_synth_setup(zkr_ctx* ctx, const zkr_r1cs_csc* r1cs, const void* toxic, void* out_a, void* out_b1,
                    void* out_b2, void* out_c, void* out_h, void* out_vk);

/* ---- setup from a powers-of-tau ceremony, phase-2 delta contributions ------------------------------------
 * Keys an operator can deploy, unlike zkr_synth_setup's: nobody has to know the toxic waste.
 *
 * Security statement.  A key made here is sound if the phase-1 ceremony's tau, alpha and beta are unknown to
 * everyone AND at least one phase-2 contributor erased their delta'.  A key straight out of zkr_setup_from_powers
 * has gamma = delta = 1 (as snarkjs's `zkey new`) and is FORGEABLE until one contribution has been applied.
 * zkr_setup_from_powers does NOT verify phase 1: neither the subgroup membership of the G2 powers nor the same-ratio
 * consistency of the powers is checked.  Check them first with zkr_powers_verify (and every phase-1 contribution
 * with zkr_powers_verify_contribution, below), or take them from a ceremony the caller already trusts.
 *
 * Phase-1 points, host memory, affine Fq-M in the binary key encoding (64 B G1, 128 B G2 = x.c0|x.c1|y.c0|y.c1);
 * n_* counts the points given, only the first are read, so a ceremony of size 2^K >= m is passed as is:
 *   tau_g1[k] = tau^k G1, n_tau_g1 >= 2m - 1      tau_g2[k] = tau^k G2, n_tau_g2 >= m
 *   alpha_tau_g1[k] = alpha tau^k G1, >= m        beta_tau_g1[k] = beta tau^k G1, >= m      beta_g2 = beta G2
 * H_(m-1) = tau^(m-1) Z(tau) G1 needs tau^(2m-1): with exactly 2m - 1 powers (a ceremony of size m) it is written as
 * infinity.  No proof uses it -- h = (AB - C)/Z has degree <= m - 2 for every satisfying witness -- but only with
 * n_tau_g1 >= 2m is the key byte-identical to zkr_synth_setup's for the same (tau, alpha, beta, 1, 1). */
typedef struct zkr_powers {
    uint32_t n_tau_g1, n_tau_g2, n_alpha_tau_g1, n_beta_tau_g1;
    const void *tau_g1, *tau_g2, *alpha_tau_g1, *beta_tau_g1, *beta_g2;
} zkr_powers;
/* The seven outputs of zkr_synth_setup (same sizes, same encoding) for gamma = delta = 1, omega = omega_m as the NTT:
 *   [L_j] = (1/m) sum_k omega^(-jk) [tau^k]    (inverse NTTs over curve points: tau_g1, alpha_tau_g1, beta_tau_g1, tau_g2)
 *   A_i = sum_j a_ij [L_j]G1,  B1_i / B2_i the same over B in G1 / G2,
 *   IC_i (i <= l) / C_i (i > l) = sum_j a_ij [beta L_j] + b_ij [alpha L_j] + c_ij [L_j],
 *   H_k = [tau^(k+m)] - [tau^k] = [tau^k Z(tau)],
 *   vk: alfa1 = alpha_tau_g1[0], beta1 = beta_tau_g1[0], delta1 = G1, beta2 = beta_g2, gamma2 = delta2 = G2.
 * Every input is checked on the host before any launch: counts, coordinates < q, points on their curve, no power at
 * infinity, R1CS rows < m and coefficients < r.  ZKR_E_INVALID otherwise; zkr_last_error names the section and index.
 * The powers themselves are not verified (G2 subgroup, same ratios): zkr_powers_verify does that. */
int zkr_setup_from_powers(zkr_ctx* ctx, const zkr_r1cs_csc* r1cs, const zkr_powers* powers, void* out_a, void* out_b1,
                          void* out_b2, void* out_c, void* out_h, void* out_vk);
#define ZKR_CONTRIB_RECORD_BYTES 96
/* One phase-2 contribution with secret delta' (32 B std form, 0 < delta' < r; NULL = drawn from getrandom).
 * pk / vk: a websnark binary proving key (zkr_pkey_load_bin's layout) and its vk block (zkr_vkey_load_bin's);
 * out_pk / out_vk: caller buffers of the same sizes.  delta1, delta2 (key header and vk block) are multiplied by
 * delta', every C and H point by delta'^-1, every other byte is copied.  out_record (96 B) is a Schnorr proof of
 * knowledge of delta' for delta1_new = delta' delta1_old:  R = k delta1_old (k from getrandom),
 *   c = SHA-256("zkr-phase2-delta" | delta1_old | delta1_new | R) as a 256-bit little-endian integer mod r
 *       (points as their 64 key bytes, Fq-M),
 *   z = k + c delta' mod r;   record = R (64 B, Fq-M) | z (32 B std).
 * delta', its inverse and k are zeroed on the host and the device before the call returns.
 * Contributions chain: call again on the output.  ZKR_E_INVALID for a malformed layout, pk and vk disagreeing on
 * delta, delta1 / delta2 not valid points, or delta' = 0 or >= r. */
int zkr_setup_contribute(zkr_ctx* ctx, const void* pk, size_t pk_len, const void* vk, size_t vk_len,
                         const void* delta32, void* out_pk, void* out_vk, void* out_record);
/* *valid = 1 iff new_pk / new_vk is old_pk / old_vk after one honest contribution proven by `record`:
 *   every byte outside delta1, delta2, C and H is unchanged; each key's header delta1 / delta2 equal its vk's;
 *   delta1 and delta2 (old and new) are valid points, not infinity, delta2 in the G2 subgroup;
 *   e(delta1_new, G2) = e(G1, delta2_new);  z delta1_old = R + c delta1_new;  every new C / H point is on the curve
 *   or infinity written as (0, R mod q);
 *   e(X_new, delta2_new) = e(X_old, delta2_old), X = sum rho_i C_i + sum sigma_k H_k with fresh 128-bit CSPRNG
 *   scalars shared by old and new (two GPU MSMs over the C|H section, host pairings).
 * ZKR_E_INVALID only for a malformed old layout or buffer sizes (both keys have pk_len / vk_len bytes). */
int zkr_setup_verify_contribution(zkr_ctx* ctx, const void* old_pk, const void* old_vk, const void* new_pk,
                                  const void* new_vk, size_t pk_len, size_t vk_len, const void* record, int* valid);

/* ---- phase 1: contributions to the powers of tau, and their verification ------------------------------------
 * The powers zkr_setup_from_powers takes, made and checked on the GPU.  Points as in zkr_powers (host memory, affine
 * Fq-M, key encoding).  Counts are free within n_tau_g1 >= 2, n_tau_g2 >= 2, n_alpha_tau_g1 >= 1, n_beta_tau_g1 >= 1,
 * each <= 2^28 (2m G1 powers for the largest m zkr_setup_from_powers takes); snarkjs's 2^(K+1) - 1 / 2^K is one case.
 * Malformed counts or NULL sections are ZKR_E_INVALID with the section named.  An empty ceremony has every point a
 * generator (tau = alpha = beta = 1). */
#define ZKR_POWERS_RECORD_BYTES 288
/* One contribution with secrets (tau', alpha', beta') = secrets96 (3 x 32 B std form, each in [1, r); NULL = each
 * drawn from getrandom, redrawn if zero).  Outputs (caller buffers of the input's counts):
 *   tau_g1'[k] = tau'^k tau_g1[k]               tau_g2'[k] = tau'^k tau_g2[k]
 *   alpha_tau_g1'[k] = alpha' tau'^k alpha_tau_g1[k]   beta_tau_g1'[k] = beta' tau'^k beta_tau_g1[k]
 *   beta_g2' = beta' beta_g2
 * so contributing to the powers of (tau, alpha, beta) gives exactly the powers of (tau tau', alpha alpha', beta beta').
 * out_record (288 B) is three Schnorr proofs of knowledge, for tau', alpha', beta' in that order, each R (64 B, Fq-M) |
 * z (32 B std).  For the secret s' with base P_old and P_new = s' P_old:  R = k P_old (k from getrandom, nonzero),
 *   c = SHA-256("zkr-phase1-" name | P_old | P_new | R) mod r  (name "tau" / "alpha" / "beta", points as their 64 key
 *       bytes, the digest a 256-bit little-endian integer),  z = k + c s' mod r,
 * with bases P_old = tau_g1[1], alpha_tau_g1[0], beta_tau_g1[0] of the input.  The format is this library's own, not
 * snarkjs's .ptau contribution.  The input is checked on the host before any launch (counts, coordinates < q, on the
 * curve, no infinity; not the G2 subgroup: that is zkr_powers_verify's job), and so are the secrets: ZKR_E_INVALID with
 * the section and index, or the secret, in the message.  The secrets, the tables of tau'^k and the nonces are zeroed on
 * the host and the device before the call returns, on error paths too. */
int zkr_powers_contribute(zkr_ctx* ctx, const zkr_powers* in, const void* secrets96, void* out_tau_g1, void* out_tau_g2,
                          void* out_alpha_tau_g1, void* out_beta_tau_g1, void* out_beta_g2, void* out_record);
/* *valid = 1 iff the powers are well formed:
 *   1. every point has coordinates < q, is on its curve and is not infinity (x encoding 0); every G2 point (tau_g2,
 *      beta_g2) is in the order-r subgroup ([r]Q = O, one GPU thread per point);
 *   2. tau_g1[0] is the G1 generator and tau_g2[0] the G2 generator, byte for byte;
 *   3. e(sum rho_k T1[k+1] + sigma_k A[k+1] + pi_k B[k+1], G2) = e(sum rho_k T1[k] + sigma_k A[k] + pi_k B[k], tau_g2[1])
 *      (T1 = tau_g1, A = alpha_tau_g1, B = beta_tau_g1; fresh 128-bit CSPRNG scalars; GPU MSMs, host pairings);
 *   4. e(G1, sum rho'_k T2[k+1]) = e(tau_g1[1], sum rho'_k T2[k])  (T2 = tau_g2);
 *   5. e(beta_tau_g1[0], G2) = e(G1, beta_g2).
 * Unlike other verdict-returning calls, *valid = 0 also sets zkr_last_error() to the first failed check, e.g.
 * "tau_g2[5] is not in the order-r subgroup" or "G1 same-ratio check failed". */
int zkr_powers_verify(zkr_ctx* ctx, const zkr_powers* p, int* valid);
/* *valid = 1 iff new_p is old_p after the contribution `record` proves:  the three old bases are valid points; each
 * proof's R is a valid point and z < r;  z P_old = R + c P_new for tau, alpha and beta;  and new_p passes every check
 * of zkr_powers_verify.  old_p is assumed verified when it was made: a transcript is checked link by link.  The first
 * failed check is in zkr_last_error(), as for zkr_powers_verify.  ZKR_E_INVALID for malformed counts or pointers, and
 * for counts that differ between old_p and new_p. */
int zkr_powers_verify_contribution(zkr_ctx* ctx, const zkr_powers* old_p, const zkr_powers* new_p, const void* record,
                                   int* valid);

/* points[i] = scalars[i] * G (group 1: G1 generator (1,2); group 2: the G2 generator of TxVerifier.sol:30-35);
 * scalars n x 32 B std form, out n x 64 / 128 B affine Fq-M; host buffers.  Workload generator for the
 * standalone MSM sweeps (BASELINE.json configs[2]). */
int zkr_synth_points(zkr_ctx* ctx, int group, const void* scalars, size_t n, void* out_points);

/* ---- test hooks (element-wise field / curve kernels; used by the parity tests) --------- */
/* field: 0 = Fq, 1 = Fr.  op: 0 mul, 1 add, 2 sub, 3 sqr, 4 inverse, 5 to_mont, 6 from_mont; sums of products with one
 * reduction: 7 = a b + (a+b)(a-b), 8 = a b - (a+b)(a-b), 9 = a b + (a+b)(a-b) + a (a-b) + (a+b) b; 10 = the dedicated
 * squaring (100 instead of 128 wide multiplies).
 * a, b, out: n x 32 B host buffers (Montgomery form operands for mul/add/sub/sqr/inverse/sums of products). */
int zkr_test_field_op(zkr_ctx* ctx, int field, int op, const void* a, const void* b, void* out, size_t n);
/* group 1/2.  op: 0 = affine+affine (via XYZZ mixed add), 1 = double, 2 = scalar mul by k[i] (32 B std),
 * 3 = 2P + 2Q through the full XYZZ add (both operands with non-trivial zz), 4 / 5 / 6 = 2P + Q through the mixed addition in
 * its plain / lazily reduced / lazily reduced + dedicated-squaring form (non-trivial zz).  Points: affine Montgomery, x == 0 = infinity; out affine Montgomery. */
int zkr_test_curve_op(zkr_ctx* ctx, int group, int op, const void* p, const void* q_or_k, void* out, size_t n);
/* white-box: copy an internal MSM work buffer of `b` to the host (what: 0 table, 1/2 keys, 3/4 vals,
 * 5 buckets, 6 result, 7 reduce partials, 8/9 boundary keys, 10/11 boundary partials). */
int zkr_test_bases_peek(const zkr_bases* b, int what, size_t offset, void* out, size_t bytes);
/* integer-pipe microbenchmarks: which: 0 = IMAD chain, 1 = IMAD.WIDE chain, 2 = Fq modmul chain,
 * 3 = XYZZ mixed-add chain, 4 = DFMA chain (FP64 pipe), 5 = DFMA + IMAD.WIDE pairs, 6 = DFMA + 64-bit
 * add pairs, 7 = 64-bit add chain; 8 = Fermat inversions, 9 = binary-Euclid inversions (full grids), 10 / 11 =
 * batched-affine additions with one inversion per thread and 16 / 64 additions (the measurement behind the
 * "batched affine" entry of DESIGN.md 4.8); 12 = lazily reduced G1 mixed-add chain, 13 / 14 = G2 mixed-add chain in its
 * plain / lazily reduced form at the MSM's 8 warps per SM, 15 = 12 with the dedicated squaring.  Returns operations per second (IMADs / modmuls / madds / pairs /
 * inversions / additions). */
int zkr_microbench(zkr_ctx* ctx, int which, int iters, double* ops_per_s, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* ZKR_H */
