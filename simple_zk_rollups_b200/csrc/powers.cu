// Phase-1 powers of tau (C-ABI: zkr_powers_contribute, zkr_powers_verify, zkr_powers_verify_contribution).  zkr.h
// states the math, the record format and the checks.
//
// The input of zkr_setup_from_powers made and checked here instead of trusted:
//   * Contribution: one thread per point multiplies it by its own scalar c tau'^k (c = 1, alpha' or beta'), taken from
//     a two-level table of powers of tau' built once per call (k_scale_points, ceremony.cuh).  The record is three
//     Schnorr proofs of knowledge (tau', alpha', beta') with host SHA-256 challenges, as phase 2's.
//   * Verification: one thread per point for range, curve and infinity, and [r]Q = O for G2; then random linear
//     combinations of consecutive powers by bucketed MSMs (zkr_msm_dev) over slices of at most 2^22 points, and host
//     pairings (verify.cu).
#include "ceremony.cuh"

using namespace zkr;

namespace {

constexpr uint32_t kMaxPowers = 1u << 28;         // 2m G1 powers for the largest domain of zkr_setup_from_powers
constexpr uint32_t kSlice = 1u << 22;             // MSM bases loaded at a time: bounds the window tables
const char* const kSecretName[3] = {"tau", "alpha", "beta"};
const char* const kTag[3] = {"zkr-phase1-tau", "zkr-phase1-alpha", "zkr-phase1-beta"};    // challenge tags

// ------------------------------------------------------------------------------------------------ contribution
// Device copy of a contribution's secrets and record scalars, std form
struct Secrets {
    Fr s[3];                            // tau', alpha', beta'
    Fr k[3];                            // Schnorr nonces
    Fr c[3], z[3];                      // challenges and responses (public)
};

__device__ __forceinline__ Fr pow_small(Fr b, uint32_t e) {
    Fr r = Fr::one();
#pragma unroll 1
    for (; e; e >>= 1) {
        if (e & 1) r = r * b;
        b = b.sqr();
    }
    return r;
}

// lo[j] = tau'^j, hi[j] = tau'^(j 2^14), Montgomery form
__global__ void k_pow_table(const Secrets* s, Fr* lo, Fr* hi) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= kTab) return;
    const Fr t = s->s[0].to_mont();
    Fr t14 = t;
#pragma unroll 1
    for (int i = 0; i < kTabLog; i++) t14 = t14.sqr();
    pow_small(t, j).store(lo + j);
    pow_small(t14, j).store(hi + j);
}

// ------------------------------------------------------------------------------------------------ verification
__device__ __forceinline__ bool in_range(const Fq& a) {
#pragma unroll
    for (int i = 7; i >= 0; i--)
        if (a.v[i] != FqParams::mod(i)) return a.v[i] < FqParams::mod(i);
    return false;
}
__device__ __forceinline__ bool in_range(const Fq2& a) { return in_range(a.c0) && in_range(a.c1); }

template <class F>
__device__ __forceinline__ F curve_b();
template <>
__device__ __forceinline__ Fq curve_b<Fq>() {          // 3
    return Fq::one() + Fq::one() + Fq::one();
}
template <>
__device__ __forceinline__ Fq2 curve_b<Fq2>() {        // 3 / (9 + u), Montgomery (verify.cu kTwistB)
    const uint32_t b0[8] = {0x77b802a8u, 0x3bf938e3u, 0x3633535du, 0x020b1b27u, 0x49755260u, 0x26b7edf0u, 0x4384a86du, 0x2514c632u};
    const uint32_t b1[8] = {0xd1dcff67u, 0x38e7ecccu, 0x93ce0d3eu, 0x65f0b37du, 0x22ac00aau, 0xd749d0ddu, 0x4a688d4du, 0x0141b9ceu};
    Fq2 b;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        b.c0.v[i] = b0[i];
        b.c1.v[i] = b1[i];
    }
    return b;
}

// *bad = min over failing points of (index << 8 | PointCheck code), the same checks and order as host_point_check:
// x == 0 is infinity, then coordinates < q, then on the curve, then (G2, `subgroup`) [r]Q = O.
template <class F>
__global__ void k_point_check(const Affine<F>* __restrict__ pts, uint32_t n, int subgroup, unsigned long long* bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Affine<F> a = Affine<F>::load_ro(pts + i);
    int code = PT_OK;
    if (a.x.is_zero()) code = PT_INFINITY;
    else if (!in_range(a.x) || !in_range(a.y)) code = PT_RANGE;
    else if (!(a.y.sqr() == a.x.sqr() * a.x + curve_b<F>())) code = PT_OFF_CURVE;
    else if (subgroup) {
        Fr r;
#pragma unroll
        for (int j = 0; j < 8; j++) r.v[j] = FrParams::mod(j);
        if (!scalar_mul(XYZZ<F>::from_affine(a), r).is_inf()) code = PT_SUBGROUP;
    }
    if (code != PT_OK) atomicMin(bad, (unsigned long long)i << 8 | (unsigned)code);
}

// acc += part (the partial sums of the MSM slices)
template <class F>
__global__ void k_xyzz_acc(XYZZ<F>* acc, const XYZZ<F>* part) {
    XYZZ<F> a = XYZZ<F>::load(acc);
    a.add(XYZZ<F>::load(part));
    a.store(acc);
}

template <class F>
__global__ void k_xyzz_key(const XYZZ<F>* p, Affine<F>* out, int n) {
    for (int i = 0; i < n; i++) store_key_point(XYZZ<F>::load(p + i), out + i);
}

// ------------------------------------------------------------------------------------------------ host
struct Section {
    const char* name;
    int group;
    const void* pts;
    uint32_t n, need;
};

void sections(const zkr_powers* p, Section out[5]) {
    out[0] = {"tau_g1", 1, p->tau_g1, p->n_tau_g1, 2};
    out[1] = {"tau_g2", 2, p->tau_g2, p->n_tau_g2, 2};
    out[2] = {"alpha_tau_g1", 1, p->alpha_tau_g1, p->n_alpha_tau_g1, 1};
    out[3] = {"beta_tau_g1", 1, p->beta_tau_g1, p->n_beta_tau_g1, 1};
    out[4] = {"beta_g2", 2, p->beta_g2, 1, 1};
}

size_t point_bytes(int group) { return group == 1 ? 64 : 128; }

// counts and pointers; ZKR_E_INVALID with the section named
int check_counts(const char* fn, const zkr_powers* p) {
    Section s[5];
    sections(p, s);
    for (const Section& x : s) {
        if (x.n < x.need || !x.pts) {
            set_error("%s: %s has %u points, %u needed", fn, x.name, x.pts ? x.n : 0u, x.need);
            return ZKR_E_INVALID;
        }
        if (x.n > kMaxPowers) {
            set_error("%s: %s has %u points, at most 2^28 allowed", fn, x.name, x.n);
            return ZKR_E_INVALID;
        }
    }
    return ZKR_OK;
}

// The first failing point of a section on the device, or index n; *code is its PointCheck code.
template <class F>
int device_point_check(zkr_ctx* ctx, cudaStream_t st, const Section& x, Affine<F>* d_pts, unsigned long long* d_bad,
                       uint32_t* idx, int* code) {
    unsigned long long bad = ~0ull;
    ZKR_CUDA(cudaMemcpyAsync(d_pts, x.pts, point_bytes(x.group) * (size_t)x.n, cudaMemcpyHostToDevice, st));
    ZKR_CUDA(cudaMemcpyAsync(d_bad, &bad, sizeof(bad), cudaMemcpyHostToDevice, st));
    ZKR_LAUNCH(ctx, k_point_check<F>, ceil_div(x.n, 128), 128, 0, st, d_pts, x.n, x.group == 2, d_bad);
    ZKR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    *idx = bad == ~0ull ? x.n : (uint32_t)(bad >> 8);
    *code = (int)(bad & 0xff);
    return ZKR_OK;
}

// Random combinations of consecutive powers over the given sections of one group, in the key encoding:
//   out[0] = sum_k rho_k P[k+1],  out[1] = sum_k rho_k P[k]   (k < n - 1 within each section, fresh 128-bit rho)
// Bases are loaded kSlice points at a time; the partial sums are added on the device.
template <class F>
int same_ratio_sums(zkr_ctx* ctx, const Section* secs, int n_secs, uint8_t* out) {
    cudaStream_t st = ctx->user_stream;         // the stream zkr_msm_dev runs on
    DevAllocs a;
    XYZZ<F>*acc, *part;
    Affine<F>* d_out;
    uint8_t* d_sc;
    ZKR_TRY(a.alloc(&acc, 2 * sizeof(XYZZ<F>)));
    ZKR_TRY(a.alloc(&part, sizeof(XYZZ<F>)));
    ZKR_TRY(a.alloc(&d_out, 2 * sizeof(Affine<F>)));
    uint32_t cap = 1;
    for (int si = 0; si < n_secs; si++) cap = std::max(cap, std::min(kSlice, secs[si].n));
    ZKR_TRY(a.alloc(&d_sc, 2 * 32 * (size_t)cap + 32));                  // zkr_msm's padding of one scalar
    ZKR_CUDA(cudaMemsetAsync(acc, 0, 2 * sizeof(XYZZ<F>), st));           // all-zero words are the identity
    std::vector<uint8_t> sc(2 * 32 * (size_t)cap), rnd(16 * (size_t)cap);
    for (int si = 0; si < n_secs; si++) {
        const Section& x = secs[si];
        uint8_t prev[16] = {};               // rho_(off - 1)
        for (uint32_t off = 0; x.n > 1 && off < x.n; off += kSlice) {     // a one-point section has no pair
            const uint32_t len = std::min(kSlice, x.n - off);
            ZKR_TRY(os_random(rnd.data(), 16 * (size_t)len));          // rho_off .. rho_(off + len - 1)
            std::fill(sc.begin(), sc.begin() + 2 * 32 * (size_t)len, 0);
            uint8_t *L = sc.data(), *R = sc.data() + 32 * (size_t)len;
            for (uint32_t j = 0; j < len; j++) {
                memcpy(L + 32 * (size_t)j, j ? &rnd[16 * (size_t)(j - 1)] : prev, 16);
                if (off + j + 1 < x.n) memcpy(R + 32 * (size_t)j, &rnd[16 * (size_t)j], 16);
            }
            memcpy(prev, &rnd[16 * (size_t)(len - 1)], 16);
            ZKR_CUDA(cudaMemcpyAsync(d_sc, sc.data(), 2 * 32 * (size_t)len, cudaMemcpyHostToDevice, st));
            zkr_bases* b = nullptr;
            ZKR_TRY(zkr_bases_load(ctx, x.group, (const uint8_t*)x.pts + point_bytes(x.group) * off, len, 0, &b));
            int rc = ZKR_OK;
            for (int side = 0; side < 2 && rc == ZKR_OK; side++) {
                rc = zkr_msm_dev(ctx, b, d_sc + 32 * (size_t)len * side, len, part);
                if (rc == ZKR_OK) {
                    k_xyzz_acc<F><<<1, 1, 0, st>>>(acc + side, part);
                    ctx->launches++;
                    const cudaError_t e = cudaPeekAtLastError();
                    if (e != cudaSuccess) rc = cuda_fail(e, "k_xyzz_acc", __FILE__, __LINE__);
                }
            }
            zkr_bases_free(b);                   // synchronises the device
            ZKR_TRY(rc);
        }
    }
    ZKR_LAUNCH(ctx, k_xyzz_key<F>, 1, 1, 0, st, acc, d_out, 2);
    ZKR_CUDA(cudaMemcpyAsync(out, d_out, 2 * sizeof(Affine<F>), cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

// zkr_powers_verify's checks; *valid = 0 with the first failed check in zkr_last_error.  Counts already checked.
int verify_powers(zkr_ctx* ctx, const char* fn, const zkr_powers* p, int* valid) {
    *valid = 0;
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    Section s[5];
    sections(p, s);
    // 1. every point in range, on its curve, not infinity; G2 in the order-r subgroup
    {
        size_t most = 0;
        for (const Section& x : s) most = std::max(most, point_bytes(x.group) * x.n);
        DevAllocs a;
        void* d_pts;
        unsigned long long* d_bad;
        ZKR_TRY(a.alloc(&d_pts, most));
        ZKR_TRY(a.alloc(&d_bad, sizeof(unsigned long long)));
        for (const Section& x : s) {
            uint32_t idx;
            int code;
            if (x.group == 1) ZKR_TRY(device_point_check<Fq>(ctx, st, x, (G1Affine*)d_pts, d_bad, &idx, &code));
            else ZKR_TRY(device_point_check<Fq2>(ctx, st, x, (G2Affine*)d_pts, d_bad, &idx, &code));
            if (idx < x.n) {
                set_error("%s: %s[%u] %s", fn, x.name, idx, point_problem(code));
                return ZKR_OK;
            }
        }
    }
    // 2. tau_g1[0] = G1, tau_g2[0] = G2
    uint8_t gen[192];
    ZKR_TRY(generators(ctx, st, gen));
    if (memcmp(p->tau_g1, gen, 64) || memcmp(p->tau_g2, gen + 64, 128)) {
        set_error("%s: %s", fn, memcmp(p->tau_g1, gen, 64) ? "tau_g1[0] is not the G1 generator" : "tau_g2[0] is not the G2 generator");
        return ZKR_OK;
    }
    const uint8_t* t1 = (const uint8_t*)p->tau_g1;
    const uint8_t* t2 = (const uint8_t*)p->tau_g2;
    // 3. e(sum rho T1[k+1] + sigma A[k+1] + pi B[k+1], G2) = e(sum rho T1[k] + sigma A[k] + pi B[k], tau_g2[1])
    {
        const Section g1s[3] = {s[0], s[2], s[3]};
        uint8_t lr[128];
        ZKR_TRY(same_ratio_sums<Fq>(ctx, g1s, 3, lr));
        const void* P[2] = {lr, lr + 64};
        const void* Q[2] = {gen + 64, t2 + 128};
        const bool neg[2] = {false, true};
        if (!host_pairing_is_one(P, neg, Q, 2)) {
            set_error("%s: G1 same-ratio check failed", fn);
            return ZKR_OK;
        }
    }
    // 4. e(G1, sum rho' T2[k+1]) = e(tau_g1[1], sum rho' T2[k])
    {
        uint8_t lr[256];
        ZKR_TRY(same_ratio_sums<Fq2>(ctx, &s[1], 1, lr));
        const void* P[2] = {gen, t1 + 64};
        const void* Q[2] = {lr, lr + 128};
        const bool neg[2] = {false, true};
        if (!host_pairing_is_one(P, neg, Q, 2)) {
            set_error("%s: G2 same-ratio check failed", fn);
            return ZKR_OK;
        }
    }
    // 5. e(beta_tau_g1[0], G2) = e(G1, beta_g2)
    {
        const void* P[2] = {p->beta_tau_g1, gen};
        const void* Q[2] = {gen + 64, p->beta_g2};
        const bool neg[2] = {false, true};
        if (!host_pairing_is_one(P, neg, Q, 2)) {
            set_error("%s: beta_tau_g1[0] and beta_g2 have different beta", fn);
            return ZKR_OK;
        }
    }
    *valid = 1;
    return ZKR_OK;
}

// The three Schnorr bases of a contribution (tau_g1[1], alpha_tau_g1[0], beta_tau_g1[0]), 64 B each
void schnorr_bases(const zkr_powers* p, uint8_t out[192]) {
    memcpy(out, (const uint8_t*)p->tau_g1 + 64, 64);
    memcpy(out + 64, p->alpha_tau_g1, 64);
    memcpy(out + 128, p->beta_tau_g1, 64);
}

}  // namespace

extern "C" int zkr_powers_contribute(zkr_ctx* ctx, const zkr_powers* in, const void* secrets96, void* out_tau_g1,
                                     void* out_tau_g2, void* out_alpha_tau_g1, void* out_beta_tau_g1, void* out_beta_g2,
                                     void* out_record) {
    static const char kFn[] = "zkr_powers_contribute";
    if (!ctx || !in || !out_tau_g1 || !out_tau_g2 || !out_alpha_tau_g1 || !out_beta_tau_g1 || !out_beta_g2 || !out_record)
        return ZKR_E_INVALID;
    ZKR_TRY(check_counts(kFn, in));
    Section s[5];
    sections(in, s);
    for (const Section& x : s) ZKR_TRY(check_section(kFn, x.name, x.group, x.pts, x.n, x.need, x.n));
    for (int j = 0; secrets96 && j < 3; j++) {
        const uint8_t* v = (const uint8_t*)secrets96 + 32 * j;
        if (is_zero32(v) || !lt_r(v)) {
            set_error("%s: %s must be in [1, r)", kFn, kSecretName[j]);
            return ZKR_E_INVALID;
        }
    }
    // host secrets: tau', alpha', beta', then the three nonces, all nonzero
    HostSecret<192> sec;
    if (secrets96) memcpy(sec.b, secrets96, 96);
    for (int j = secrets96 ? 3 : 0; j < 6; j++) ZKR_TRY(draw_nonzero(sec.b + 32 * j));
    uint8_t p_old[192], small[3 * 64];          // Schnorr bases, then R
    schnorr_bases(in, p_old);

    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    // the secrets, the nonces and the tables of tau'^k are secret buffers; the point buffers hold only public values
    // (inputs, outputs and R)
    DevAllocs a;
    Secrets* d_sec;
    Fr* d_tab;                                  // lo | hi
    G1Affine* d_r;
    void* d_pts;
    ZKR_TRY(a.alloc_secret(&d_sec, sizeof(Secrets), st));
    ZKR_TRY(a.alloc_secret(&d_tab, 2 * sizeof(Fr) * kTab, st));
    ZKR_CUDA(cudaMemcpyAsync(d_sec, sec.b, sizeof(sec.b), cudaMemcpyHostToDevice, st));      // s[3] | k[3]
    size_t most = 0;
    for (const Section& x : s) most = std::max(most, point_bytes(x.group) * x.n);
    ZKR_TRY(a.alloc(&d_pts, most));
    ZKR_TRY(a.alloc(&d_r, 3 * sizeof(G1Affine)));
    const Fr *lo = d_tab, *hi = d_tab + kTab;
    ZKR_LAUNCH(ctx, k_pow_table, kTab / 128, 128, 0, st, d_sec, d_tab, d_tab + kTab);
    // tau_g1, tau_g2 by tau'^k; alpha_tau_g1 by alpha' tau'^k; beta_tau_g1 by beta' tau'^k; beta_g2 by beta'
    void* const outs[5] = {out_tau_g1, out_tau_g2, out_alpha_tau_g1, out_beta_tau_g1, out_beta_g2};
    const Fr* coef[5] = {nullptr, nullptr, d_sec->s + 1, d_sec->s + 2, d_sec->s + 2};
    for (int i = 0; i < 5; i++) {
        const Section& x = s[i];
        const size_t bytes = point_bytes(x.group) * x.n;
        ZKR_CUDA(cudaMemcpyAsync(d_pts, x.pts, bytes, cudaMemcpyHostToDevice, st));
        if (x.group == 1)
            ZKR_LAUNCH(ctx, k_scale_points<Fq>, ceil_div(x.n, 128), 128, 0, st, (G1Affine*)d_pts, x.n, lo, hi, coef[i]);
        else
            ZKR_LAUNCH(ctx, k_scale_points<Fq2>, ceil_div(x.n, 128), 128, 0, st, (G2Affine*)d_pts, x.n, lo, hi, coef[i]);
        ZKR_CUDA(cudaMemcpyAsync(outs[i], d_pts, bytes, cudaMemcpyDeviceToHost, st));
        ZKR_CUDA(cudaStreamSynchronize(st));
    }
    // R_j = k_j P_old_j
    ZKR_CUDA(cudaMemcpyAsync(d_r, p_old, sizeof(p_old), cudaMemcpyHostToDevice, st));
    for (int j = 0; j < 3; j++)
        ZKR_LAUNCH(ctx, k_scale_points<Fq>, 1, 1, 0, st, d_r + j, (size_t)1, nullptr, nullptr, d_sec->k + j);
    ZKR_CUDA(cudaMemcpyAsync(small, d_r, sizeof(small), cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    uint8_t p_new[192], c[96];
    memcpy(p_new, (const uint8_t*)out_tau_g1 + 64, 64);
    memcpy(p_new + 64, out_alpha_tau_g1, 64);
    memcpy(p_new + 128, out_beta_tau_g1, 64);
    for (int j = 0; j < 3; j++) challenge(kTag[j], p_old + 64 * j, p_new + 64 * j, small + 64 * j, c + 32 * j);
    ZKR_CUDA(cudaMemcpyAsync(d_sec->c, c, sizeof(c), cudaMemcpyHostToDevice, st));
    ZKR_LAUNCH(ctx, k_schnorr_z, 1, 1, 0, st, d_sec->s, d_sec->k, d_sec->c, d_sec->z, 3);
    uint8_t* rec = (uint8_t*)out_record;
    for (int j = 0; j < 3; j++) {
        memcpy(rec + 96 * j, small + 64 * j, 64);
        ZKR_CUDA(cudaMemcpyAsync(rec + 96 * j + 64, d_sec->z + j, 32, cudaMemcpyDeviceToHost, st));
    }
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

extern "C" int zkr_powers_verify(zkr_ctx* ctx, const zkr_powers* p, int* valid) {
    if (!ctx || !p || !valid) return ZKR_E_INVALID;
    *valid = 0;
    ZKR_TRY(check_counts("zkr_powers_verify", p));
    return verify_powers(ctx, "zkr_powers_verify", p, valid);
}

extern "C" int zkr_powers_verify_contribution(zkr_ctx* ctx, const zkr_powers* old_p, const zkr_powers* new_p,
                                              const void* record, int* valid) {
    static const char kFn[] = "zkr_powers_verify_contribution";
    if (!ctx || !old_p || !new_p || !record || !valid) return ZKR_E_INVALID;
    *valid = 0;
    ZKR_TRY(check_counts(kFn, old_p));
    ZKR_TRY(check_counts(kFn, new_p));
    if (old_p->n_tau_g1 != new_p->n_tau_g1 || old_p->n_tau_g2 != new_p->n_tau_g2 ||
        old_p->n_alpha_tau_g1 != new_p->n_alpha_tau_g1 || old_p->n_beta_tau_g1 != new_p->n_beta_tau_g1) {
        set_error("%s: old and new powers have different counts", kFn);
        return ZKR_E_INVALID;
    }
    static const char* const kBase[3] = {"tau_g1[1]", "alpha_tau_g1[0]", "beta_tau_g1[0]"};
    uint8_t p_old[192], p_new[192];
    schnorr_bases(old_p, p_old);
    schnorr_bases(new_p, p_new);
    const uint8_t* rec = (const uint8_t*)record;
    for (int j = 0; j < 3; j++) {
        int code = host_point_check(1, p_old + 64 * j, false);
        if (code != PT_OK) {
            set_error("%s: old %s %s", kFn, kBase[j], point_problem(code));
            return ZKR_OK;
        }
        if ((code = host_point_check(1, p_new + 64 * j, false)) != PT_OK) {
            set_error("%s: %s %s", kFn, kBase[j], point_problem(code));
            return ZKR_OK;
        }
        if ((code = host_point_check(1, rec + 96 * j, false)) != PT_OK) {
            set_error("%s: the %s proof's R %s", kFn, kSecretName[j], point_problem(code));
            return ZKR_OK;
        }
        if (!lt_r(rec + 96 * j + 64)) {
            set_error("%s: the %s proof's z is >= r", kFn, kSecretName[j]);
            return ZKR_OK;
        }
    }
    // z P_old = R + c P_new, for tau, alpha, beta
    {
        DeviceGuard g(ctx->device);
        for (int j = 0; j < 3; j++) {
            bool ok;
            const uint8_t* R = rec + 96 * j;
            ZKR_TRY(schnorr_holds(ctx, ctx->s[0], kTag[j], p_old + 64 * j, p_new + 64 * j, R, R + 64, &ok));
            if (!ok) {
                set_error("%s: the %s proof of knowledge does not hold", kFn, kSecretName[j]);
                return ZKR_OK;
            }
        }
    }
    return verify_powers(ctx, kFn, new_p, valid);
}
