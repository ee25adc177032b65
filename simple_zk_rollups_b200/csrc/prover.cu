// Groth16 prove on one B200: proving-key residency, sparse A_T/B_T, H pipeline, five MSMs, assembly.
//
// C-ABI: zkr_pkey_load_bin / zkr_pkey_free / zkr_pkey_info / zkr_prove / zkr_prove_dev / zkr_prove_batch.
// Replaces, for /root/reference/operator/src/snarks/common.ts:
//   :28  binarifyProvingKey(provingKey) on every proof  -> zkr_pkey_load_bin once per circuit
//   :29  wasmBn128.groth16GenProof(witnessBin, pkBin)   -> zkr_prove
// Math: SURVEY.md Appendix B.2/B.3 (oracle: oracle/groth16.py gen_proof).
//
//   pi_a = alfa1 + sum w_i A_i + r delta1            one G1 MSM over [A.., alfa1, delta1] x [w.., 1, r]
//   pib1 = beta1 + sum w_i B1_i + s delta1           one G1 MSM over [B1.., beta1, delta1] x [w.., 1, s]
//   pi_b = beta2 + sum w_i B2_i + s delta2           one G2 MSM over [B2.., beta2, delta2] x [w.., 1, s]
//   pi_c = sum_{i>l} w_i C_i - rs delta1  (one MSM)  +  sum h_j hExps_j (one MSM)  +  s pi_a + r pib1
// The blinding terms ride inside the MSMs as extra bases, so the only scalar multiplications left
// are s*pi_a and r*pib1 (two threads, overlapped with the G2 / C / H MSMs on other streams).
#include <sys/random.h>
#include <unistd.h>

#include <cstdlib>
#include <cstring>
#include <thread>

#include "comm_iface.cuh"
#include "ec.cuh"
#include "msm_iface.cuh"
#include "ntt_iface.cuh"

using namespace zkr;

struct zkr_pkey {
    zkr_ctx* ctx = nullptr;
    uint32_t n_vars = 0, n_public = 0, domain_size = 0;
    int log_m = 0;
    int rank = 0, world = 1;       // world > 1: the five base sets hold this rank's point range only
    uint64_t h_lo = 0;             // first h coefficient (bit-reversed order) of this rank's hExps slice
    uint64_t h_count = 0;          // size of that slice; 0 = this rank is outside the H group (shard_plan) and skips the H chain
    // polsA / polsB as CSR by constraint row (coefficients Fr-M exactly as in the key)
    uint32_t *a_ptr = nullptr, *a_sig = nullptr, *b_ptr = nullptr, *b_sig = nullptr;
    Fr *a_coef = nullptr, *b_coef = nullptr;
    uint64_t nnz_a = 0, nnz_b = 0;
    zkr_bases *A = nullptr, *B1 = nullptr, *B2 = nullptr, *C = nullptr, *H = nullptr;
    // per-proof work buffers (one proof in flight per key)
    Fr* wext = nullptr;      // [w_0..w_{n-1}, 1, r, s, -rs]  standard form
    Fr *at = nullptr, *bt = nullptr, *st = nullptr, *h = nullptr;
    char* res = nullptr;     // XYZZ results: A(128) B1(128) C(128) H(128) T1(128) T2(128) B2(256)
    char* proof = nullptr;   // 256 B affine standard form
    int* err = nullptr;      // device flag: witness[0] != 1 or r/s out of range
    char* rs_dev = nullptr;  // 64 B staging for (r | s)
    void* pinned = nullptr;  // 256 + 64 B pinned host staging
    // zkr_prove_batch: second witness buffer + upload events, so that witness i+1 is uploaded while proof i runs
    Fr* wext2 = nullptr;
    cudaEvent_t ev_up[2] = {};
    cudaEvent_t ev[19] = {};   // 0..15 stage timing (zkr_stats), 16..18 sharded tail (ZKR_TIMELINE)
    // B1' and B2' take the same scalars through the same compaction map and window plan (B1_i is the point at infinity
    // exactly when B2_i is): one digit extraction + radix sort, done on pi_b's stream, serves both MSMs
    bool share_b_sort = false;
    cudaEvent_t ev_b2_sorted = nullptr;
    size_t bytes = 0;
};

namespace {

enum { R_A = 0, R_B1 = 128, R_C = 256, R_H = 384, R_T1 = 512, R_T2 = 640, R_B2 = 768, R_TOTAL = 1024 };

// A_T[c] = sum_k coef[k] * w[sig[k]]  (coef Montgomery x w standard -> standard)
__device__ __forceinline__ void sparse_lc(uint32_t c, const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ sig,
                                          const Fr* __restrict__ coef, const Fr* __restrict__ w, Fr* __restrict__ out) {
    Fr acc = Fr::zero();
    const uint32_t e = ptr[c + 1];
    for (uint32_t k = ptr[c]; k < e; k++) acc = acc + Fr::load_ro(coef + k) * Fr::load_ro(w + sig[k]);
    acc.store(out + c);
}
__global__ void k_sparse_lc(const uint32_t* __restrict__ a_ptr, const uint32_t* __restrict__ a_sig,
                            const Fr* __restrict__ a_coef, const uint32_t* __restrict__ b_ptr,
                            const uint32_t* __restrict__ b_sig, const Fr* __restrict__ b_coef,
                            const Fr* __restrict__ w, Fr* __restrict__ at, Fr* __restrict__ bt, uint32_t m) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    const bool isb = blockIdx.y != 0;
    sparse_lc(c, isb ? b_ptr : a_ptr, isb ? b_sig : a_sig, isb ? b_coef : a_coef, w, isb ? bt : at);
}
// batched: proof blockIdx.z reads its witness at w + z wstride and writes its A_T / B_T at at / bt + z m
__global__ void k_sparse_lc_many(const uint32_t* __restrict__ a_ptr, const uint32_t* __restrict__ a_sig,
                                 const Fr* __restrict__ a_coef, const uint32_t* __restrict__ b_ptr,
                                 const uint32_t* __restrict__ b_sig, const Fr* __restrict__ b_coef,
                                 const Fr* __restrict__ w, size_t wstride, Fr* __restrict__ at, Fr* __restrict__ bt, uint32_t m) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    const bool isb = blockIdx.y != 0;
    const size_t j = blockIdx.z;
    sparse_lc(c, isb ? b_ptr : a_ptr, isb ? b_sig : a_sig, isb ? b_coef : a_coef, w + j * wstride, (isb ? bt : at) + j * m);
}

// wext[n] = 1, wext[n+1] = r, wext[n+2] = s, wext[n+3] = -(r s) mod r_order; returns 1 if r or s >= r, 2 if w_0 != 1
__device__ __forceinline__ int prep_scalars(Fr* wext, uint32_t n, const Fr* rs) {
    Fr r = Fr::load(rs), s = Fr::load(rs + 1);
    int e = 0;
    if (!r.in_range() || !s.in_range()) e = 1;
    Fr one = Fr::zero();
    one.v[0] = 1;
    if (Fr::load(wext) != one) e = 2;
    Fr rsm = (r.to_mont() * s.to_mont()).from_mont();
    one.store(wext + n);
    r.store(wext + n + 1);
    s.store(wext + n + 2);
    rsm.neg().store(wext + n + 3);
    return e;
}
__global__ void k_prep_scalars(Fr* wext, uint32_t n, const Fr* rs, int* err) {
    const int e = prep_scalars(wext, n, rs);
    if (e) *err = e;
}
// batched: one thread per proof, extended witness j at wext + j (n + 4), (r | s) at rs + 2 j; err[j] |= 1 (r / s), 2 (w_0)
__global__ void k_prep_scalars_many(Fr* wext, uint32_t n, const Fr* rs, int* err, int k) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const int e = prep_scalars(wext + (size_t)j * (n + 4), n, rs + 2 * j);
    if (e) atomicOr(err + j, e == 2 ? 2 : 1);
}

// every witness value must be < r (signals that touch no base are read by no MSM)
__global__ void k_witness_range(const Fr* __restrict__ w, uint32_t n, int* err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !Fr::load_ro(w + i).in_range()) *err = 1;
}
// batched: proof blockIdx.y, witness at w + y wstride; err[y] |= 1
__global__ void k_witness_range_many(const Fr* __restrict__ w, uint32_t n, size_t wstride, int* err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !Fr::load_ro(w + blockIdx.y * wstride + i).in_range()) atomicOr(err + blockIdx.y, 1);
}

// block 0: T1 = s * pi_a ; block 1: T2 = r * pib1.
// The 254-step doubling chain is the only serial part of a scalar multiplication; everything else is taken
// off it: lane 0 of warp 0 only doubles and publishes 2^i P in shared memory, lane 0 of warps 1..7 add the
// published multiples whose scalar bit is set (bit i belongs to warp 1 + i mod 7) at their own pace, thread 0
// adds the seven partial sums.  Latency 254 doublings + ~8 additions instead of 254 doublings + ~127 additions
// (1.3 ms -> 0.8 ms); it is on the critical path of the small circuits (tx.circom, withdraw.circom), hidden behind
// the G2 MSM at 2^20 and above.  One active lane per warp on purpose: divergent lanes of one warp would serialise.
constexpr int kBlindWarps = 8;
__device__ __forceinline__ void blind_mul(char* res, const Fr* wext, uint32_t n, bool second) {
    extern __shared__ unsigned char blind_sm[];
    G1XYZZ* chain = reinterpret_cast<G1XYZZ*>(blind_sm);            // [256]
    G1XYZZ* part = chain + 256;                                      // [kBlindWarps]
    __shared__ volatile int ready;                                   // chain[0 .. ready) are published
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const Fr k = Fr::load(wext + n + (second ? 1 : 2));
    int top = 255;
    while (top >= 0 && !((k.v[top >> 5] >> (top & 31)) & 1)) top--;
    if (threadIdx.x == 0) ready = 0;
    __syncthreads();
    if (lane == 0) {
        if (warp == 0) {
            G1XYZZ base = G1XYZZ::load(res + (second ? R_B1 : R_A));
#pragma unroll 1
            for (int i = 0; i <= top; i++) {
                chain[i] = base;
                __threadfence_block();
                ready = i + 1;
                if (i < top) base = base.dbl();
            }
        } else {
            G1XYZZ acc = G1XYZZ::identity();
#pragma unroll 1
            for (int i = warp - 1; i <= top; i += kBlindWarps - 1) {
                if (!((k.v[i >> 5] >> (i & 31)) & 1)) continue;
                while (ready <= i) {
                }
                __threadfence_block();
                G1XYZZ d = chain[i];
                acc.add(d);
            }
            part[warp] = acc;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        G1XYZZ acc = part[1];
#pragma unroll 1
        for (int w = 2; w < kBlindWarps; w++) {
            G1XYZZ d = part[w];
            acc.add(d);
        }
        acc.store(res + (second ? R_T2 : R_T1));
    }
}
__global__ void __launch_bounds__(32 * kBlindWarps) k_blind_muls(char* res, const Fr* wext, uint32_t n) {
    blind_mul(res, wext, n, blockIdx.x != 0);
}
// batched: blocks 2 j and 2 j + 1 blind proof j (results at res + j R_TOTAL, extended witness at wext + j (n + 4))
__global__ void __launch_bounds__(32 * kBlindWarps) k_blind_muls_many(char* res, const Fr* wext, uint32_t n) {
    const uint32_t j = blockIdx.x >> 1;
    blind_mul(res + (size_t)j * R_TOTAL, wext + (size_t)j * (n + 4), n, blockIdx.x & 1);
}
constexpr size_t kBlindSmem = sizeof(G1XYZZ) * (256 + kBlindWarps);

// block 0: pi_a, block 1: pi_b, block 2: pi_c = C + H + T1 + T2; affine, standard form
// Three single-thread blocks, nothing left to overlap them: the inversion is the whole kernel, so it is the binary
// extended Euclid of fp_inv.cuh (faster than the a^(p-2) ladder here: profiles/r01_small_circuits_finish_ab.json).
__device__ __forceinline__ void finish(const char* res, char* proof, unsigned part) {
    if (part == 0) {
        const G1XYZZ p = G1XYZZ::load(res + R_A);
        G1Affine a = p.to_affine_vartime();
        a.x.from_mont().store(proof);
        a.y.from_mont().store(proof + 32);
    } else if (part == 1) {
        const G2XYZZ p = G2XYZZ::load(res + R_B2);
        G2Affine a = p.to_affine_vartime();
        a.x.from_mont().store(proof + 64);
        a.y.from_mont().store(proof + 128);
    } else {
        G1XYZZ c = G1XYZZ::load(res + R_C);
#pragma unroll 1
        for (int i = 0; i < 3; i++) c.add(G1XYZZ::load(res + (i == 0 ? R_H : (i == 1 ? R_T1 : R_T2))));
        G1Affine a = c.to_affine_vartime();
        a.x.from_mont().store(proof + 192);
        a.y.from_mont().store(proof + 224);
    }
}
__global__ void k_finish(const char* res, char* proof) { finish(res, proof, blockIdx.x); }
// batched: blocks 3 j .. 3 j + 2 assemble proof j
__global__ void k_finish_many(const char* res, char* proof) {
    const uint32_t j = blockIdx.x / 3;
    finish(res + (size_t)j * R_TOTAL, proof + (size_t)j * ZKR_PROOF_BYTES, blockIdx.x - 3 * j);
}

// sharded prove: res[e] = sum over ranks of the gathered partial results (block e: B2 in G2; A, B1, C, H, T1, T2 in
// G1; every rank blinds its own partials, so the blinding terms are partial sums too)
__global__ void k_sum_res(const char* slots, int world, char* res) {
    const int offs[7] = {R_B2, R_A, R_B1, R_C, R_H, R_T1, R_T2};
    const int off = offs[blockIdx.x];
    if (blockIdx.x > 0) {
        G1XYZZ acc = G1XYZZ::load(slots + off);
#pragma unroll 1
        for (int r = 1; r < world; r++) acc.add(G1XYZZ::load(slots + (size_t)r * kCommSlotBytes + off));
        acc.store(res + off);
    } else {
        G2XYZZ acc = G2XYZZ::load(slots + off);
#pragma unroll 1
        for (int r = 1; r < world; r++) acc.add(G2XYZZ::load(slots + (size_t)r * kCommSlotBytes + off));
        acc.store(res + off);
    }
}

struct PkView {
    uint32_t n, l, m, pA, pB, pPA, pPB1, pPB2, pPC, pPH;
};

bool is_pow2(uint32_t x) { return x && !(x & (x - 1)); }

// walk one pols section (binarify.ts:104-113): per signal u32 count, then count x (u32 row, 32 B coef)
int pols_to_csr(const uint8_t* buf, size_t len, size_t off, size_t end, uint32_t n, uint32_t m,
                std::vector<uint32_t>& ptr, std::vector<uint32_t>& sig, std::vector<uint8_t>& coef) {
    ptr.assign((size_t)m + 1, 0);
    size_t o = off;
    uint64_t nnz = 0;
    for (uint32_t s = 0; s < n; s++) {
        if (o + 4 > end) return ZKR_E_BADKEY;
        uint32_t k;
        memcpy(&k, buf + o, 4);
        o += 4;
        if ((uint64_t)k * 36 > end - o) return ZKR_E_BADKEY;
        for (uint32_t j = 0; j < k; j++) {
            uint32_t row;
            memcpy(&row, buf + o + 36ull * j, 4);
            if (row >= m) return ZKR_E_BADKEY;
            ptr[row + 1]++;
        }
        o += 36ull * k;
        nnz += k;
    }
    if (o != end) return ZKR_E_BADKEY;
    for (uint32_t c = 0; c < m; c++) ptr[c + 1] += ptr[c];
    sig.resize(nnz);
    coef.resize(nnz * 32);
    std::vector<uint32_t> cur(ptr.begin(), ptr.end() - 1);
    o = off;
    for (uint32_t s = 0; s < n; s++) {
        uint32_t k;
        memcpy(&k, buf + o, 4);
        o += 4;
        for (uint32_t j = 0; j < k; j++) {
            uint32_t row;
            memcpy(&row, buf + o, 4);
            const uint32_t d = cur[row]++;
            sig[d] = s;
            memcpy(&coef[32ull * d], buf + o + 4, 32);
            o += 36;
        }
    }
    (void)len;
    return ZKR_OK;
}

int upload(const void* h, size_t bytes, void** d, cudaStream_t st, size_t* total) {
    ZKR_CUDA(cudaMalloc(d, bytes ? bytes : 16));
    if (bytes) ZKR_CUDA(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    *total += bytes;
    return ZKR_OK;
}

void pkey_release(zkr_pkey* pk) {
    if (!pk) return;
    void* ps[] = {pk->a_ptr, pk->a_sig, pk->a_coef, pk->b_ptr, pk->b_sig, pk->b_coef, pk->wext, pk->at, pk->bt,
                  pk->st, pk->h, pk->res, pk->proof, pk->err, pk->rs_dev};
    for (void* p : ps) cudaFree(p);
    if (pk->wext2) cudaFree(pk->wext2);
    for (auto& e : pk->ev_up)
        if (e) cudaEventDestroy(e);
    if (pk->pinned) cudaFreeHost(pk->pinned);
    for (auto& e : pk->ev)
        if (e) cudaEventDestroy(e);
    if (pk->ev_b2_sorted) cudaEventDestroy(pk->ev_b2_sorted);
    zkr_bases* bs[] = {pk->A, pk->B1, pk->B2, pk->C, pk->H};
    for (zkr_bases* b : bs) bases_release(b);
    delete pk;
}

}  // namespace

// [lo, hi) of `total` entries owned by `rank` (balanced to within one entry; mirrors sharding.point_range)
static void shard_range(uint64_t total, int rank, int world, uint64_t* lo, uint64_t* hi) {
    const uint64_t base = total / world, rem = total % world;
    *lo = rank * base + ((uint64_t)rank < rem ? rank : rem);
    *hi = *lo + base + ((uint64_t)rank < rem ? 1 : 0);
}

// How one proof is split over `world` ranks (SURVEY.md 8(e) "single-proof latency split": one part of the box runs
// sparse LC + H pipeline + the hExps MSM, the rest runs the witness MSMs; websnark fans the same calls out to web
// workers, operator/src/snarks/common.ts:29).  The H pipeline does not shard at rollup sizes, so replicating it on every
// rank costs 1.7 ms per rank.  Instead only the first g_h ranks (the "H group") run it, each followed by 1/g_h of the
// hExps MSM; the witness MSMs (A', B1', B2', C') are split by point range with WEIGHTS: a fraction x of the points
// to each H-group rank, y to each of the others, chosen so that every rank gets the same modelled work
//     H-group rank:  P + MH / g_h + x W        other rank:  y W         g_h x + (world - g_h) y = 1
// in units of one G1 point of a 2^20 MSM (P = H pipeline, MH = m, W = n (2 + 2.4) + nc; a G2 point costs 2.4 G1
// points, the H pipeline 0.85 m: profiles/r02_launch_shares.md).  ZKR_SHARD_TASKS=0 restores the uniform split with
// the H pipeline on every rank; every rank of a job must see the same value.
struct ShardPlan {
    int g_h = 1;
    double x = 1, y = 1;
    bool uniform = true;
};
static ShardPlan shard_plan(int world, uint64_t n, uint64_t nc, uint64_t m) {
    ShardPlan p;
    p.g_h = world;
    p.x = p.y = 1.0 / world;
    const char* e = getenv("ZKR_SHARD_TASKS");
    if (world == 1 || (e && atoi(e) == 0)) return p;
    p.uniform = false;
    p.g_h = world <= 2 ? 1 : world / 2;
    const double P = 0.85 * (double)m, MH = (double)m, W = (double)n * 4.4 + (double)nc;
    const double T = (p.g_h * P + MH + W) / world;
    p.x = (T - P - MH / p.g_h) / W;
    if (p.x < 0.06) p.x = 0;                       // not worth four more latency chains beside the H chain
    if (p.x * p.g_h > 1) p.x = 1.0 / p.g_h;
    p.y = (1.0 - p.g_h * p.x) / (world - p.g_h);
    return p;
}
// rank's [lo, hi) of the witness MSMs' `total` points under the plan (cumulative weights, last rank ends at total)
static void plan_range(const ShardPlan& p, uint64_t total, int rank, int world, uint64_t* lo, uint64_t* hi) {
    if (p.uniform) return shard_range(total, rank, world, lo, hi);
    auto cum = [&](int r) -> uint64_t {
        if (r >= world) return total;
        const double f = r <= p.g_h ? r * p.x : p.g_h * p.x + (r - p.g_h) * p.y;
        const uint64_t v = (uint64_t)(f * (double)total);
        return v > total ? total : v;
    };
    *lo = cum(rank);
    *hi = cum(rank + 1);
}

static int pkey_load(zkr_ctx* ctx, const void* vbuf, size_t len, int rank, int world, zkr_pkey** out) {
    if (!ctx || !vbuf || !out || world < 1 || rank < 0 || rank >= world) return ZKR_E_INVALID;
    *out = nullptr;
    const uint8_t* buf = (const uint8_t*)vbuf;
    if (len < 488) {
        set_error("proving key too short (%zu bytes)", len);
        return ZKR_E_BADKEY;
    }
    PkView v;
    memcpy(&v, buf, 40);
    const uint64_t n = v.n, l = v.l, m = v.m;
    bool ok = n >= 1 && l + 1 <= n && is_pow2(v.m) && m >= 2 && m <= (1u << 27) && v.pA == 488 && v.pA <= v.pB &&
              v.pB <= v.pPA && v.pPA <= len;
    ok = ok && (uint64_t)v.pPA + 64 * n == v.pPB1 && (uint64_t)v.pPB1 + 64 * n == v.pPB2 &&
         (uint64_t)v.pPB2 + 128 * n == v.pPC && (uint64_t)v.pPC + 64 * (n - l - 1) == v.pPH &&
         (uint64_t)v.pPH + 64 * m == len;
    if (!ok) {
        set_error("proving key header inconsistent (nVars=%u nPublic=%u domainSize=%u len=%zu)", v.n, v.l, v.m, len);
        return ZKR_E_BADKEY;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    zkr_pkey* pk = new zkr_pkey();
    pk->ctx = ctx;
    pk->n_vars = v.n;
    pk->n_public = v.l;
    pk->domain_size = v.m;
    pk->rank = rank;
    pk->world = world;
    while ((1u << pk->log_m) < v.m) pk->log_m++;
    uint64_t lo = 0, hi = 0;
    const ShardPlan plan = shard_plan(world, n, n - l - 1, m);
    int rc = ZKR_OK;
#define PK_TRY(expr)              \
    do {                          \
        rc = (expr);              \
        if (rc != ZKR_OK) {       \
            pkey_release(pk);     \
            return rc;            \
        }                         \
    } while (0)
    {   // polsA, polsB -> CSR
        std::vector<uint32_t> ptr, sig;
        std::vector<uint8_t> coef;
        rc = pols_to_csr(buf, len, v.pA, v.pB, v.n, v.m, ptr, sig, coef);
        if (rc != ZKR_OK) {
            set_error("polsA section malformed");
            pkey_release(pk);
            return rc;
        }
        pk->nnz_a = sig.size();
        PK_TRY(upload(ptr.data(), ptr.size() * 4, (void**)&pk->a_ptr, st, &pk->bytes));
        PK_TRY(upload(sig.data(), sig.size() * 4, (void**)&pk->a_sig, st, &pk->bytes));
        PK_TRY(upload(coef.data(), coef.size(), (void**)&pk->a_coef, st, &pk->bytes));
        rc = pols_to_csr(buf, len, v.pB, v.pPA, v.n, v.m, ptr, sig, coef);
        if (rc != ZKR_OK) {
            set_error("polsB section malformed");
            pkey_release(pk);
            return rc;
        }
        pk->nnz_b = sig.size();
        PK_TRY(upload(ptr.data(), ptr.size() * 4, (void**)&pk->b_ptr, st, &pk->bytes));
        PK_TRY(upload(sig.data(), sig.size() * 4, (void**)&pk->b_sig, st, &pk->bytes));
        PK_TRY(upload(coef.data(), coef.size(), (void**)&pk->b_coef, st, &pk->bytes));
    }
    const uint8_t *alfa1 = buf + 40, *beta1 = buf + 104, *delta1 = buf + 168, *beta2 = buf + 232, *delta2 = buf + 360;
    const uint32_t N = v.n;
    {   // A' = [A.., alfa1, delta1] x [w.., 1, r]
        std::vector<char> pts(64ull * (n + 2));
        memcpy(pts.data(), buf + v.pPA, 64 * n);
        memcpy(&pts[64 * n], alfa1, 64);
        memcpy(&pts[64 * (n + 1)], delta1, 64);
        std::vector<uint32_t> sidx(n + 2);
        for (uint32_t i = 0; i < N + 2; i++) sidx[i] = i;            // n -> 1, n+1 -> r
        pk->A = bases_alloc();
        bases_set_group(pk->A, 1);
        plan_range(plan, n + 2, rank, world, &lo, &hi);
        PK_TRY(bases_build_g1(ctx, pk->A, pts.data() + 64 * lo, hi - lo, 0, st, sidx.data() + lo));
        // B1' = [B1.., beta1, delta1] x [w.., 1, s]
        memcpy(pts.data(), buf + v.pPB1, 64 * n);
        memcpy(&pts[64 * n], beta1, 64);
        sidx[N + 1] = N + 2;                                          // s
        pk->B1 = bases_alloc();
        bases_set_group(pk->B1, 1);
        PK_TRY(bases_build_g1(ctx, pk->B1, pts.data() + 64 * lo, hi - lo, 0, st, sidx.data() + lo));
        // B2' = [B2.., beta2, delta2] x [w.., 1, s]
        std::vector<char> pts2(128ull * (n + 2));
        memcpy(pts2.data(), buf + v.pPB2, 128 * n);
        memcpy(&pts2[128 * n], beta2, 128);
        memcpy(&pts2[128 * (n + 1)], delta2, 128);
        pk->B2 = bases_alloc();
        bases_set_group(pk->B2, 2);
        PK_TRY(bases_build_g2(ctx, pk->B2, pts2.data() + 128 * lo, hi - lo, 0, st, sidx.data() + lo));
    }
    {   // C' = [C_{l+1}.., delta1] x [w_{l+1}.., -rs]
        const uint64_t nc = n - l - 1;
        std::vector<char> pts(64ull * (nc + 1));
        memcpy(pts.data(), buf + v.pPC, 64 * nc);
        memcpy(&pts[64 * nc], delta1, 64);
        std::vector<uint32_t> sidx(nc + 1);
        for (uint64_t i = 0; i < nc; i++) sidx[i] = (uint32_t)(l + 1 + i);
        sidx[nc] = N + 3;
        pk->C = bases_alloc();
        bases_set_group(pk->C, 1);
        plan_range(plan, nc + 1, rank, world, &lo, &hi);
        PK_TRY(bases_build_g1(ctx, pk->C, pts.data() + 64 * lo, hi - lo, 0, st, sidx.data() + lo));
    }
    {   // H: hExps permuted to bit-reversed order (the H pipeline leaves h bit-reversed)
        std::vector<char> pts(64ull * m);
        const int lg = pk->log_m;
        for (uint64_t p = 0; p < m; p++) {
            uint32_t j = 0;
            for (int b = 0; b < lg; b++) j |= ((p >> b) & 1u) << (lg - 1 - b);
            memcpy(&pts[64 * p], buf + v.pPH + 64ull * j, 64);
        }
        pk->H = bases_alloc();
        bases_set_group(pk->H, 1);
        if (rank < plan.g_h) shard_range(m, rank, plan.g_h, &lo, &hi);
        else lo = hi = 0;                                             // not in the H group: no H pipeline, no hExps slice
        pk->h_lo = lo;
        pk->h_count = hi - lo;
        PK_TRY(bases_build_g1(ctx, pk->H, pts.data() + 64 * lo, hi - lo, 0, st, nullptr));
    }
    // work buffers
    auto dmalloc = [&](void** p, size_t bytes) -> int {
        ZKR_CUDA(cudaMalloc(p, bytes));
        pk->bytes += bytes;
        return ZKR_OK;
    };
    PK_TRY(dmalloc((void**)&pk->wext, 32 * (n + 4)));
    PK_TRY(dmalloc((void**)&pk->at, 32 * m));
    PK_TRY(dmalloc((void**)&pk->bt, 32 * m));
    PK_TRY(dmalloc((void**)&pk->st, 32 * m));
    PK_TRY(dmalloc((void**)&pk->h, 32 * m));
    PK_TRY(dmalloc((void**)&pk->res, R_TOTAL));
    PK_TRY(dmalloc((void**)&pk->proof, ZKR_PROOF_BYTES));
    PK_TRY(dmalloc((void**)&pk->err, sizeof(int)));
    PK_TRY(dmalloc((void**)&pk->rs_dev, 64));
    if (cudaMallocHost(&pk->pinned, 512) != cudaSuccess) {
        pkey_release(pk);
        return ZKR_E_NOMEM;
    }
    cudaMemsetAsync(pk->err, 0, sizeof(int), st);
    for (auto& e : pk->ev) cudaEventCreate(&e);
    cudaEventCreateWithFlags(&pk->ev_b2_sorted, cudaEventDisableTiming);
    pk->share_b_sort = bases_share_sort(pk->B1, pk->B2);
    NttTables* t;
    PK_TRY(ntt_get_tables(ctx, pk->log_m, &t));
    zkr_bases* bs[] = {pk->A, pk->B1, pk->B2, pk->C, pk->H};
    for (zkr_bases* b : bs) {
        uint64_t bb = 0;
        bases_info(b, nullptr, nullptr, nullptr, &bb);
        pk->bytes += bb;
    }
    cudaStreamSynchronize(st);
#undef PK_TRY
    *out = pk;
    return ZKR_OK;
}

extern "C" int zkr_pkey_load_bin(zkr_ctx* ctx, const void* vbuf, size_t len, zkr_pkey** out) {
    return pkey_load(ctx, vbuf, len, 0, 1, out);
}

extern "C" int zkr_shard_ranges(int world, int rank, uint64_t n_vars, uint64_t n_public, uint64_t domain_size,
                                uint64_t* out6) {
    if (!out6 || world < 1 || rank < 0 || rank >= world || n_vars < n_public + 1) return ZKR_E_INVALID;
    const uint64_t nc = n_vars - n_public - 1;
    const ShardPlan plan = shard_plan(world, n_vars, nc, domain_size);
    plan_range(plan, n_vars + 2, rank, world, &out6[0], &out6[1]);
    plan_range(plan, nc + 1, rank, world, &out6[2], &out6[3]);
    if (rank < plan.g_h) shard_range(domain_size, rank, plan.g_h, &out6[4], &out6[5]);
    else out6[4] = out6[5] = 0;
    return ZKR_OK;
}

extern "C" int zkr_pkey_load_bin_sharded(zkr_ctx* ctx, const void* vbuf, size_t len, int rank, int world, zkr_pkey** out) {
    return pkey_load(ctx, vbuf, len, rank, world, out);
}

extern "C" void zkr_pkey_free(zkr_pkey* pk) {
    if (!pk) return;
    DeviceGuard g(pk->ctx->device);
    cudaDeviceSynchronize();
    pkey_release(pk);
}

extern "C" int zkr_pkey_info(const zkr_pkey* pk, uint32_t* n_vars, uint32_t* n_public, uint32_t* domain_size,
                             uint64_t* device_bytes) {
    if (!pk) return ZKR_E_INVALID;
    if (n_vars) *n_vars = pk->n_vars;
    if (n_public) *n_public = pk->n_public;
    if (domain_size) *domain_size = pk->domain_size;
    if (device_bytes) *device_bytes = pk->bytes;
    return ZKR_OK;
}

// Queue one proof: witness already in pk->wext[0..n), (r|s) in pk->rs_dev.  Result -> d_proof.
static int prove_enqueue(zkr_ctx* ctx, const zkr_pkey* pk, char* d_proof, bool timed, zkr_comm* comm = nullptr,
                         Fr* wext = nullptr) {
    const uint32_t n = pk->n_vars, m = pk->domain_size;
    if (!wext) wext = pk->wext;
    cudaStream_t us = ctx->user_stream;
    cudaEvent_t const* ev = pk->ev;
    ZKR_LAUNCH(ctx, k_prep_scalars, 1, 1, 0, us, wext, n, (const Fr*)pk->rs_dev, pk->err);
    ZKR_LAUNCH(ctx, k_witness_range, ceil_div(n, 256), 256, 0, us, wext, n, pk->err);
    const bool par = !ctx->serial;
    // one stream per chain: s[0] = H, s[1] = A, s[2] = B1, s[3] = B2, s[4] = C
    if (par) ZKR_TRY(ctx->fork(5));
    cudaStream_t sH = par ? ctx->s[0] : us, sA = par ? ctx->s[1] : us, sB1 = par ? ctx->s[2] : us,
                 sB2 = par ? ctx->s[3] : us, sC = par ? ctx->s[4] : us;
    const uint32_t* w = (const uint32_t*)wext;
    // heaviest first: the G2 MSM costs ~3 G1 MSMs
    if (timed) cudaEventRecord(ev[6], sB2);
    ZKR_TRY(msm_run_g2(ctx, sB2, pk->B2, w, pk->res + R_B2, nullptr, pk->ev_b2_sorted));
    if (timed) cudaEventRecord(ev[7], sB2);
    // H chain: sparse LC, H pipeline, hExps MSM
    if (timed) cudaEventRecord(ev[0], sH);
    if (pk->h_count != 0) {
        ZKR_LAUNCH(ctx, k_sparse_lc, dim3(ceil_div(m, 128), 2), 128, 0, sH, pk->a_ptr, pk->a_sig, pk->a_coef, pk->b_ptr,
                   pk->b_sig, pk->b_coef, wext, pk->at, pk->bt, m);
        if (timed) cudaEventRecord(ev[1], sH);
        ZKR_TRY(h_pipeline(ctx, sH, pk->at, pk->bt, pk->st, pk->h, pk->log_m, true));
        if (timed) cudaEventRecord(ev[2], sH);
        ZKR_TRY(msm_run_g1(ctx, sH, pk->H, (const uint32_t*)(pk->h + pk->h_lo), pk->res + R_H));
    } else {   // a rank outside the H group of a sharded proof (shard_plan)
        if (timed) cudaEventRecord(ev[1], sH);
        if (timed) cudaEventRecord(ev[2], sH);
        ZKR_CUDA(cudaMemsetAsync(pk->res + R_H, 0, 128, sH));   // the identity (ZZ = 0)
    }
    if (timed) cudaEventRecord(ev[3], sH);
    // A, then s * pi_a
    if (timed) cudaEventRecord(ev[4], sA);
    ZKR_TRY(msm_run_g1(ctx, sA, pk->A, w, pk->res + R_A));
    if (timed) cudaEventRecord(ev[5], sA);
    if (timed) cudaEventRecord(ev[8], sB1);
    if (pk->share_b_sort) ZKR_CUDA(cudaStreamWaitEvent(sB1, pk->ev_b2_sorted, 0));
    ZKR_TRY(msm_run_g1(ctx, sB1, pk->B1, w, pk->res + R_B1, pk->share_b_sort ? pk->B2 : nullptr));
    if (timed) cudaEventRecord(ev[9], sB1);
    if (timed) cudaEventRecord(ev[10], sC);
    ZKR_TRY(msm_run_g1(ctx, sC, pk->C, w, pk->res + R_C));
    if (timed) cudaEventRecord(ev[11], sC);
    // the two blinding scalar multiplications T1 = s * pi_a, T2 = r * pib1 need A and B1.  A sharded proof's results are
    // partial sums over this rank's point ranges; scalar multiplication is linear, so each rank blinds its own partial
    // A / B1 behind the A chain (off the critical H chain) and the gather sums seven partials.
    if (par) {
        ZKR_CUDA(cudaEventRecord(ctx->ev_join[2], sB1));
        ZKR_CUDA(cudaStreamWaitEvent(sA, ctx->ev_join[2], 0));
    }
    ZKR_LAUNCH(ctx, k_blind_muls, 2, 32 * kBlindWarps, kBlindSmem, sA, pk->res, wext, n);
    if (par) ZKR_TRY(ctx->join(5));
    if (comm && comm->world > 1) {
        if (timed) cudaEventRecord(ev[16], us);
        int parity = 0;
        ZKR_TRY(comm_allgather_small(comm, us, pk->res, R_TOTAL, &parity));
        if (timed) cudaEventRecord(ev[17], us);
        ZKR_LAUNCH(ctx, k_sum_res, 7, 1, 0, us, comm_gather_slot(comm, comm->rank, parity, 0), comm->world, pk->res);
        if (timed) cudaEventRecord(ev[18], us);
    }
    if (timed) cudaEventRecord(ev[12], us);
    ZKR_LAUNCH(ctx, k_finish, 3, 1, 0, us, (const char*)pk->res, d_proof);
    if (timed) cudaEventRecord(ev[13], us);
    return ZKR_OK;
}

static int check_range_flags(zkr_ctx* ctx, const zkr_pkey* pk) {
    int e = 0;
    ZKR_CUDA(cudaMemcpyAsync(&e, pk->err, sizeof(int), cudaMemcpyDeviceToHost, ctx->user_stream));
    ZKR_CUDA(cudaStreamSynchronize(ctx->user_stream));
    int any = e;
    const zkr_bases* bs[] = {pk->A, pk->B1, pk->B2, pk->C, pk->H};
    for (const zkr_bases* b : bs) {
        int be = 0;
        ZKR_TRY(bases_range_error(b, ctx->user_stream, &be));
        any |= be;
    }
    if (e) ZKR_CUDA(cudaMemsetAsync(pk->err, 0, sizeof(int), ctx->user_stream));
    if (any) {
        set_error(e == 2 ? "witness[0] must be 1" : "a witness value or blinding scalar is >= r");
        return ZKR_E_WITNESS_RANGE;
    }
    return ZKR_OK;
}

// Blinding scalar for a caller that passed NULL: uniform in [0, r) from the OS CSPRNG (getrandom), by rejection on
// 254-bit draws -- what websnark's groth16GenProof does internally.  The snarkjs debug mode (r = s = 0, deterministic,
// not zero-knowledge) has to be asked for with explicit zero buffers.
int zkr::os_random(void* out, size_t bytes) {
    size_t got = 0;
    while (got < bytes) {
        ssize_t k = getrandom((char*)out + got, bytes - got, 0);
        if (k < 0) {
            set_error("getrandom failed: no entropy source for the random scalars");
            return ZKR_E_INVALID;
        }
        got += (size_t)k;
    }
    return ZKR_OK;
}
const uint32_t zkr::kRModulus[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u,
                                    0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
int zkr::draw_scalar(void* out32) {
    for (int tries = 0; tries < 256; tries++) {
        uint32_t v[8];
        ZKR_TRY(os_random(v, sizeof(v)));
        v[7] &= 0x3fffffffu;
        bool less = false;
        for (int i = 7; i >= 0; i--) {
            if (v[i] != kRModulus[i]) {
                less = v[i] < kRModulus[i];
                break;
            }
        }
        if (less) {
            memcpy(out32, v, 32);
            explicit_bzero(v, sizeof(v));       // the scalar may be a secret (a phase-2 delta'): no stack copy survives
            return ZKR_OK;
        }
    }
    return ZKR_E_INVALID;
}
static int stage_blinding(char* dst64, const void* r32, const void* s32) {
    if (r32) memcpy(dst64, r32, 32);
    else ZKR_TRY(draw_scalar(dst64));
    if (s32) memcpy(dst64 + 32, s32, 32);
    else ZKR_TRY(draw_scalar(dst64 + 32));
    return ZKR_OK;
}

// Forget range flags left behind by earlier asynchronous proofs nobody checked (zkr_prove_dev without
// zkr_prove_check): a blocking call must report on ITS inputs only.
static int clear_range_flags(zkr_ctx* ctx, const zkr_pkey* pk) {
    ZKR_CUDA(cudaMemsetAsync(pk->err, 0, sizeof(int), ctx->user_stream));
    const zkr_bases* bs[] = {pk->A, pk->B1, pk->B2, pk->C, pk->H};
    for (const zkr_bases* b : bs) ZKR_TRY(bases_range_clear(b, ctx->user_stream));
    return ZKR_OK;
}

static int prove_host(zkr_ctx* ctx, const zkr_pkey* pk, const void* witness, size_t n_signals, const void* r32,
                      const void* s32, void* out_proof, zkr_stats* stats, zkr_comm* comm) {
    if (!ctx || !pk || !witness || !out_proof || pk->ctx != ctx) return ZKR_E_INVALID;
    if (pk->world != (comm ? comm->world : 1) || (comm && (comm->rank != pk->rank || !comm->connected))) {
        set_error("key was loaded for rank %d of %d; use the matching zkr_prove / zkr_prove_sharded call", pk->rank, pk->world);
        return ZKR_E_INVALID;
    }
    if (n_signals != pk->n_vars) {
        set_error("witness has %zu signals, key expects %u", n_signals, pk->n_vars);
        return ZKR_E_INVALID;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t us = ctx->user_stream;
    const uint64_t launches0 = ctx->launches;
    char* pin = (char*)pk->pinned;
    ZKR_TRY(stage_blinding(pin + 256, r32, s32));
    cudaEvent_t const* ev = pk->ev;
    ZKR_TRY(clear_range_flags(ctx, pk));
    cudaEventRecord(ev[14], us);
    ZKR_CUDA(cudaMemcpyAsync(pk->wext, witness, 32ull * pk->n_vars, cudaMemcpyHostToDevice, us));
    ZKR_CUDA(cudaMemcpyAsync(pk->rs_dev, pin + 256, 64, cudaMemcpyHostToDevice, us));
    ZKR_TRY(prove_enqueue(ctx, pk, pk->proof, true, comm));
    ZKR_CUDA(cudaMemcpyAsync(pin, pk->proof, ZKR_PROOF_BYTES, cudaMemcpyDeviceToHost, us));
    cudaEventRecord(ev[15], us);
    ZKR_CUDA(cudaStreamSynchronize(us));
    if (comm) ZKR_TRY(comm_check(comm, us));
    int rc = check_range_flags(ctx, pk);
    if (rc != ZKR_OK) return rc;
    memcpy(out_proof, pin, ZKR_PROOF_BYTES);
    zkr_stats s = {};
    auto el = [&](int a, int b) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ev[a], ev[b]);
        return ms;
    };
    s.total_ms = el(14, 15);
    s.h2d_ms = 0;   // included in total; the copy is queued ahead of the first kernel on the same stream
    s.lc_ms = el(0, 1);
    s.ntt_ms = el(1, 2);
    s.msm_h_ms = el(2, 3);
    s.msm_a_ms = el(4, 5);
    s.msm_b2_ms = el(6, 7);
    s.msm_b1_ms = el(8, 9);
    s.msm_c_ms = el(10, 11);
    s.assemble_ms = el(12, 13);
    s.kernel_launches = ctx->launches - launches0;
    // ZKR_TIMELINE=1 (measurement knob): offsets of every stage event from the start of the call, on stderr --
    // the zkr_stats durations do not say when a chain started (tools/gpu_jobs/r02_sharded_timeline.sh)
    static const bool timeline = getenv("ZKR_TIMELINE") && atoi(getenv("ZKR_TIMELINE")) != 0;
    if (timeline) {
        static const char* names[14] = {"lc0", "lc1", "ntt1", "msm_h1", "a0", "a1", "b2_0", "b2_1", "b1_0", "b1_1",
                                        "c0", "c1", "tail0", "finish1"};
        char line[640];
        int o = snprintf(line, sizeof line, "zkr timeline rank %d/%d total %.3f:", pk->rank, pk->world, s.total_ms);
        for (int i = 0; i < 14; i++) o += snprintf(line + o, sizeof line - o, " %s=%.3f", names[i], el(14, i));
        if (comm && comm->world > 1)
            o += snprintf(line + o, sizeof line - o, " joined=%.3f gathered=%.3f summed=%.3f", el(14, 16), el(14, 17), el(14, 18));
        line[o++] = '\n';
        if (write(2, line, (size_t)o) < 0) {   // one write per line: the ranks of a torchrun job share the pipe
        }
    }
    ctx->last_stats = s;
    if (stats) *stats = s;
    return ZKR_OK;
}

extern "C" int zkr_prove(zkr_ctx* ctx, const zkr_pkey* pk, const void* witness, size_t n_signals, const void* r32,
                         const void* s32, void* out_proof, zkr_stats* stats) {
    return prove_host(ctx, pk, witness, n_signals, r32, s32, out_proof, stats, nullptr);
}

extern "C" int zkr_prove_sharded(zkr_comm* comm, const zkr_pkey* pk, const void* witness, size_t n_signals,
                                 const void* r32, const void* s32, void* out_proof, zkr_stats* stats) {
    if (!comm) return ZKR_E_INVALID;
    if (!r32 || !s32) {
        set_error("zkr_prove_sharded: r32 and s32 are required (every rank must use the same blinding scalars)");
        return ZKR_E_INVALID;
    }
    return prove_host(comm->ctx, pk, witness, n_signals, r32, s32, out_proof, stats, comm);
}

extern "C" int zkr_prove_dev(zkr_ctx* ctx, const zkr_pkey* pk, const void* d_witness, size_t n_signals,
                             const void* r32, const void* s32, void* d_out_proof) {
    if (!ctx || !pk || !d_witness || !d_out_proof || pk->ctx != ctx || n_signals != pk->n_vars || pk->world != 1)
        return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    cudaStream_t us = ctx->user_stream;
    char* pin = (char*)pk->pinned;
    // the staging words are re-used per call: wait for the previous call's copy to have been consumed
    ZKR_CUDA(cudaStreamSynchronize(us));
    ZKR_TRY(stage_blinding(pin + 256, r32, s32));
    ZKR_CUDA(cudaMemcpyAsync(pk->wext, d_witness, 32ull * pk->n_vars, cudaMemcpyDeviceToDevice, us));
    ZKR_CUDA(cudaMemcpyAsync(pk->rs_dev, pin + 256, 64, cudaMemcpyHostToDevice, us));
    return prove_enqueue(ctx, pk, (char*)d_out_proof, false);
}

// zkr_prove_dev is asynchronous and cannot return ZKR_E_WITNESS_RANGE itself: the device-side flags (witness value or
// blinding scalar >= r, witness[0] != 1) stay set until they are read here.  Synchronises the ctx stream, reports and
// clears them: ZKR_OK means every zkr_prove_dev on this key since the last check had valid inputs.
extern "C" int zkr_prove_check(zkr_ctx* ctx, const zkr_pkey* pk) {
    if (!ctx || !pk || pk->ctx != ctx) return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    return check_range_flags(ctx, pk);
}

// All proofs assigned to one context, pipelined: while proof k runs, the witness of proof k+1 is uploaded into the
// other witness buffer on the context's copy stream (s[5]); the host only waits for proof k's 256 bytes and flags.
static int prove_batch_ctx(zkr_ctx* ctx, const zkr_pkey* pk, const void* const* witnesses, size_t n_signals,
                           int first, int stride, int n_proofs, const void* rs32, void* out_proofs) {
    if (!ctx || !pk || pk->ctx != ctx || pk->world != 1) {
        set_error("zkr_prove_batch: keys[i] must be a non-sharded key loaded on ctxs[i]");
        return ZKR_E_INVALID;
    }
    if (n_signals != pk->n_vars) {
        set_error("witness has %zu signals, key expects %u", n_signals, pk->n_vars);
        return ZKR_E_INVALID;
    }
    if (first >= n_proofs) return ZKR_OK;
    DeviceGuard g(ctx->device);
    zkr_pkey* mpk = const_cast<zkr_pkey*>(pk);
    const size_t wbytes = 32ull * pk->n_vars;
    if (!mpk->wext2) {
        ZKR_CUDA(cudaMalloc((void**)&mpk->wext2, 32ull * (pk->n_vars + 4)));
        mpk->bytes += 32ull * (pk->n_vars + 4);
        for (auto& e : mpk->ev_up) ZKR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    Fr* buf[2] = {pk->wext, pk->wext2};
    cudaStream_t us = ctx->user_stream, cs = ctx->s[kNumStreams - 1];
    char* pin = (char*)pk->pinned;
    for (int i = first; i < n_proofs; i += stride)
        if (!witnesses[i]) {
            set_error("zkr_prove_batch: witnesses[%d] is null", i);
            return ZKR_E_INVALID;
        }
    // everything queued on the user stream so far (a previous proof on this key) must be done with buf[0]
    ZKR_TRY(clear_range_flags(ctx, pk));
    ZKR_CUDA(cudaStreamSynchronize(us));
    ZKR_CUDA(cudaMemcpyAsync(buf[0], witnesses[first], wbytes, cudaMemcpyHostToDevice, cs));
    ZKR_CUDA(cudaEventRecord(pk->ev_up[0], cs));
    int k = 0;
    for (int i = first; i < n_proofs; i += stride, k++) {
        const int cur = k & 1;
        ZKR_TRY(stage_blinding(pin + 256, rs32 ? (const char*)rs32 + 64ull * i : nullptr,
                               rs32 ? (const char*)rs32 + 64ull * i + 32 : nullptr));
        ZKR_CUDA(cudaStreamWaitEvent(us, pk->ev_up[cur], 0));
        ZKR_CUDA(cudaMemcpyAsync(pk->rs_dev, pin + 256, 64, cudaMemcpyHostToDevice, us));
        ZKR_TRY(prove_enqueue(ctx, pk, pk->proof, false, nullptr, buf[cur]));
        ZKR_CUDA(cudaMemcpyAsync(pin, pk->proof, ZKR_PROOF_BYTES, cudaMemcpyDeviceToHost, us));
        if (i + stride < n_proofs) {      // proof k-1, the last reader of buf[cur ^ 1], was waited for below
            ZKR_CUDA(cudaMemcpyAsync(buf[cur ^ 1], witnesses[i + stride], wbytes, cudaMemcpyHostToDevice, cs));
            ZKR_CUDA(cudaEventRecord(pk->ev_up[cur ^ 1], cs));
        }
        ZKR_CUDA(cudaStreamSynchronize(us));
        int rc = check_range_flags(ctx, pk);
        if (rc != ZKR_OK) {
            cudaStreamSynchronize(cs);
            return rc;
        }
        memcpy((char*)out_proofs + (size_t)ZKR_PROOF_BYTES * i, pin, ZKR_PROOF_BYTES);
    }
    ZKR_CUDA(cudaStreamSynchronize(cs));
    return ZKR_OK;
}

extern "C" int zkr_prove_batch(zkr_ctx* const* ctxs, const zkr_pkey* const* pks, int n_ctx,
                               const void* const* witnesses, size_t n_signals, int n_proofs, const void* rs32,
                               void* out_proofs) {
    if (!ctxs || !pks || n_ctx < 1 || (!witnesses && n_proofs) || n_proofs < 0 || (!out_proofs && n_proofs)) return ZKR_E_INVALID;
    std::vector<int> rcs(n_ctx, ZKR_OK);
    std::vector<std::string> msgs(n_ctx);
    if (n_ctx == 1) {
        return prove_batch_ctx(ctxs[0], pks[0], witnesses, n_signals, 0, 1, n_proofs, rs32, out_proofs);
    }
    std::vector<std::thread> th;
    for (int c = 0; c < n_ctx; c++) {
        th.emplace_back([&, c]() {
            int rc = prove_batch_ctx(ctxs[c], pks[c], witnesses, n_signals, c, n_ctx, n_proofs, rs32, out_proofs);
            if (rc != ZKR_OK) {
                rcs[c] = rc;
                msgs[c] = zkr_last_error();
            }
        });
    }
    for (auto& t : th) t.join();
    for (int c = 0; c < n_ctx; c++)
        if (rcs[c] != ZKR_OK) {
            set_error("proof batch failed on context %d: %s", c, msgs[c].c_str());
            return rcs[c];
        }
    return ZKR_OK;
}

// ------------------------------------------------------------------------------------------------ many proofs, one pass
// zkr_prove_many: the k proofs of one call go through every stage together (DESIGN.md 4.10).  Each buffer holds k
// per-proof slices back to back: extended witnesses at stride n + 4, A_T / B_T / S / h at stride m, results at stride
// R_TOTAL.  The five MSMs key proof j's digits j * nbuckets + |digit| - 1 over the key's own tables; every kernel takes
// the proof index from its grid, so the launch count does not depend on k.
struct zkr_many {
    zkr_ctx* ctx = nullptr;
    const zkr_pkey* pk = nullptr;
    int max_proofs = 0;
    MsmMany *A = nullptr, *B1 = nullptr, *B2 = nullptr, *C = nullptr, *H = nullptr;
    Fr* wext = nullptr;                       // k x (n + 4)
    Fr *at = nullptr, *bt = nullptr, *st = nullptr, *h = nullptr;   // k x m each
    char* res = nullptr;                      // k x R_TOTAL
    char* proof = nullptr;                    // k x 256
    Fr* rs_dev = nullptr;                     // k x 64
    int* err = nullptr;                       // k flags: 1 a witness value or r / s >= r, 2 witness[0] != 1
    char* pinned = nullptr;                   // k x (256 proof + 64 r|s + 4 flag)
    cudaEvent_t ev_b2_sorted = nullptr;
    size_t bytes = 0;
};

static void many_release(zkr_many* mw) {
    if (!mw) return;
    for (MsmMany* w : {mw->A, mw->B1, mw->B2, mw->C, mw->H}) msm_many_free(w);
    void* ps[] = {mw->wext, mw->at, mw->bt, mw->st, mw->h, mw->res, mw->proof, mw->rs_dev, mw->err};
    for (void* p : ps) cudaFree(p);
    if (mw->pinned) cudaFreeHost(mw->pinned);
    if (mw->ev_b2_sorted) cudaEventDestroy(mw->ev_b2_sorted);
    delete mw;
}

extern "C" int zkr_many_create(zkr_ctx* ctx, const zkr_pkey* pk, int max_proofs, zkr_many** out) {
    if (!ctx || !pk || !out || pk->ctx != ctx || max_proofs < 1) return ZKR_E_INVALID;
    *out = nullptr;
    if (pk->world != 1) {
        set_error("zkr_many_create: the key is sharded (rank %d of %d); batches need a whole key", pk->rank, pk->world);
        return ZKR_E_UNSUPPORTED;
    }
    if (pk->log_m < 3) {
        set_error("zkr_many_create: domain size %u; the batched H pipeline needs at least 8", pk->domain_size);
        return ZKR_E_UNSUPPORTED;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    zkr_many* mw = new zkr_many();
    mw->ctx = ctx;
    mw->pk = pk;
    mw->max_proofs = max_proofs;
    const size_t k = (size_t)max_proofs, n = pk->n_vars, m = pk->domain_size;
    int rc = ZKR_OK;
#define MANY_TRY(expr)             \
    do {                           \
        rc = (expr);               \
        if (rc != ZKR_OK) {        \
            many_release(mw);      \
            return rc;             \
        }                          \
    } while (0)
    // B1' borrows B2''s sort when the two share one (as prove_enqueue does)
    const bool share = pk->share_b_sort;
    struct { const zkr_bases* b; MsmMany** w; bool sorts; } sets[] = {
        {pk->A, &mw->A, true}, {pk->B1, &mw->B1, !share}, {pk->B2, &mw->B2, true}, {pk->C, &mw->C, true}, {pk->H, &mw->H, true}};
    for (auto& s : sets) {
        rc = msm_many_alloc(s.b, max_proofs, s.sorts, st, s.w);
        if (rc != ZKR_OK) {
            if (rc == ZKR_E_UNSUPPORTED) {
                std::string why = zkr_last_error();
                set_error("zkr_many_create: %s", why.c_str());
            }
            many_release(mw);
            return rc;
        }
        mw->bytes += msm_many_bytes(*s.w);
    }
    auto dmalloc = [&](void** p, size_t bytes) -> int {
        ZKR_CUDA(cudaMalloc(p, bytes));
        mw->bytes += bytes;
        return ZKR_OK;
    };
    MANY_TRY(dmalloc((void**)&mw->wext, 32 * k * (n + 4)));
    MANY_TRY(dmalloc((void**)&mw->at, 32 * k * m));
    MANY_TRY(dmalloc((void**)&mw->bt, 32 * k * m));
    MANY_TRY(dmalloc((void**)&mw->st, 32 * k * m));
    MANY_TRY(dmalloc((void**)&mw->h, 32 * k * m));
    MANY_TRY(dmalloc((void**)&mw->res, R_TOTAL * k));
    MANY_TRY(dmalloc((void**)&mw->proof, ZKR_PROOF_BYTES * k));
    MANY_TRY(dmalloc((void**)&mw->rs_dev, 64 * k));
    MANY_TRY(dmalloc((void**)&mw->err, sizeof(int) * k));
    if (cudaMallocHost((void**)&mw->pinned, (ZKR_PROOF_BYTES + 64 + sizeof(int)) * k) != cudaSuccess) {
        cudaGetLastError();
        many_release(mw);
        set_error("zkr_many_create: no pinned host memory for %d proofs", max_proofs);
        return ZKR_E_NOMEM;
    }
    if (cudaEventCreateWithFlags(&mw->ev_b2_sorted, cudaEventDisableTiming) != cudaSuccess) {
        many_release(mw);
        return ZKR_E_CUDA;
    }
#undef MANY_TRY
    *out = mw;
    return ZKR_OK;
}

extern "C" void zkr_many_free(zkr_many* mw) {
    if (!mw) return;
    DeviceGuard g(mw->ctx->device);
    cudaDeviceSynchronize();
    many_release(mw);
}

extern "C" int zkr_many_info(const zkr_many* mw, int* max_proofs, uint64_t* device_bytes) {
    if (!mw) return ZKR_E_INVALID;
    if (max_proofs) *max_proofs = mw->max_proofs;
    if (device_bytes) *device_bytes = mw->bytes;
    return ZKR_OK;
}

static bool below_r(const uint8_t* v32) {
    for (int i = 7; i >= 0; i--) {
        uint32_t x;
        memcpy(&x, v32 + 4 * i, 4);
        if (x != kRModulus[i]) return x < kRModulus[i];
    }
    return false;
}

extern "C" int zkr_prove_many(zkr_ctx* ctx, zkr_many* mw, const void* witnesses, size_t n_signals, int n_proofs,
                              const void* rs32, void* out_proofs) {
    if (!ctx || !mw || !witnesses || !out_proofs || mw->ctx != ctx) return ZKR_E_INVALID;
    const zkr_pkey* pk = mw->pk;
    if (n_proofs < 1 || n_proofs > mw->max_proofs) {
        set_error("zkr_prove_many: %d proofs, the workspace holds 1 .. %d", n_proofs, mw->max_proofs);
        return ZKR_E_INVALID;
    }
    if (n_signals != pk->n_vars) {
        set_error("witness has %zu signals, key expects %u", n_signals, pk->n_vars);
        return ZKR_E_INVALID;
    }
    const int k = n_proofs;
    const uint32_t n = pk->n_vars, m = pk->domain_size;
    const size_t ws = (size_t)n + 4;
    char* pin_proof = mw->pinned;
    char* pin_rs = pin_proof + (size_t)ZKR_PROOF_BYTES * mw->max_proofs;
    int* pin_err = (int*)(pin_rs + 64ull * mw->max_proofs);
    if (rs32) {
        for (int j = 0; j < k; j++)
            for (int h = 0; h < 2; h++)
                if (!below_r((const uint8_t*)rs32 + 64ull * j + 32 * h)) {
                    set_error("proof %d: blinding scalar %s is >= r", j, h ? "s" : "r");
                    return ZKR_E_INVALID;
                }
        memcpy(pin_rs, rs32, 64ull * k);
    } else {
        for (int j = 0; j < k; j++) ZKR_TRY(stage_blinding(pin_rs + 64ull * j, nullptr, nullptr));
    }
    DeviceGuard g(ctx->device);
    cudaStream_t us = ctx->user_stream;
    ZKR_CUDA(cudaMemsetAsync(mw->err, 0, sizeof(int) * k, us));
    // k witnesses into their n + 4 slots: one strided copy
    ZKR_CUDA(cudaMemcpy2DAsync(mw->wext, 32 * ws, witnesses, 32ull * n, 32ull * n, k, cudaMemcpyHostToDevice, us));
    ZKR_CUDA(cudaMemcpyAsync(mw->rs_dev, pin_rs, 64ull * k, cudaMemcpyHostToDevice, us));
    ZKR_LAUNCH(ctx, k_prep_scalars_many, ceil_div(k, 64), 64, 0, us, mw->wext, n, (const Fr*)mw->rs_dev, mw->err, k);
    ZKR_LAUNCH(ctx, k_witness_range_many, dim3(ceil_div(n, 256), k), 256, 0, us, mw->wext, n, ws, mw->err);
    // the streams and the order of prove_enqueue: s[0] = H, s[1] = A, s[2] = B1, s[3] = B2, s[4] = C
    const bool par = !ctx->serial;
    if (par) ZKR_TRY(ctx->fork(5));
    cudaStream_t sH = par ? ctx->s[0] : us, sA = par ? ctx->s[1] : us, sB1 = par ? ctx->s[2] : us,
                 sB2 = par ? ctx->s[3] : us, sC = par ? ctx->s[4] : us;
    const uint32_t* w = (const uint32_t*)mw->wext;
    const bool share = pk->share_b_sort;
    ZKR_TRY(msm_many_run(ctx, sB2, pk->B2, mw->B2, k, w, ws, mw->res + R_B2, R_TOTAL, nullptr,
                         share ? mw->ev_b2_sorted : nullptr));
    ZKR_LAUNCH(ctx, k_sparse_lc_many, dim3(ceil_div(m, 128), 2, k), 128, 0, sH, pk->a_ptr, pk->a_sig, pk->a_coef, pk->b_ptr,
               pk->b_sig, pk->b_coef, mw->wext, ws, mw->at, mw->bt, m);
    ZKR_TRY(h_pipeline_many(ctx, sH, mw->at, mw->bt, mw->st, mw->h, pk->log_m, k));
    ZKR_TRY(msm_many_run(ctx, sH, pk->H, mw->H, k, (const uint32_t*)mw->h, m, mw->res + R_H, R_TOTAL));
    ZKR_TRY(msm_many_run(ctx, sA, pk->A, mw->A, k, w, ws, mw->res + R_A, R_TOTAL));
    if (share) ZKR_CUDA(cudaStreamWaitEvent(sB1, mw->ev_b2_sorted, 0));
    ZKR_TRY(msm_many_run(ctx, sB1, pk->B1, mw->B1, k, w, ws, mw->res + R_B1, R_TOTAL, share ? mw->B2 : nullptr));
    ZKR_TRY(msm_many_run(ctx, sC, pk->C, mw->C, k, w, ws, mw->res + R_C, R_TOTAL));
    if (par) {
        ZKR_CUDA(cudaEventRecord(ctx->ev_join[2], sB1));
        ZKR_CUDA(cudaStreamWaitEvent(sA, ctx->ev_join[2], 0));
    }
    ZKR_LAUNCH(ctx, k_blind_muls_many, 2 * k, 32 * kBlindWarps, kBlindSmem, sA, mw->res, mw->wext, n);
    if (par) ZKR_TRY(ctx->join(5));
    ZKR_LAUNCH(ctx, k_finish_many, 3 * k, 1, 0, us, (const char*)mw->res, mw->proof);
    ZKR_CUDA(cudaMemcpyAsync(pin_proof, mw->proof, (size_t)ZKR_PROOF_BYTES * k, cudaMemcpyDeviceToHost, us));
    ZKR_CUDA(cudaMemcpyAsync(pin_err, mw->err, sizeof(int) * k, cudaMemcpyDeviceToHost, us));
    ZKR_CUDA(cudaStreamSynchronize(us));
    for (int j = 0; j < k; j++)
        if (pin_err[j]) {
            set_error(pin_err[j] & 2 ? "proof %d: witness[0] must be 1" : "proof %d: a witness value is >= r", j);
            return ZKR_E_WITNESS_RANGE;
        }
    memcpy(out_proofs, pin_proof, (size_t)ZKR_PROOF_BYTES * k);
    return ZKR_OK;
}
