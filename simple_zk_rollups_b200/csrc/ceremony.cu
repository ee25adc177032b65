// Groth16 setup from a powers-of-tau ceremony and phase-2 delta contributions (C-ABI: zkr_setup_from_powers,
// zkr_setup_contribute, zkr_setup_verify_contribution).  zkr.h states the math, the encodings and what a key made
// here is sound under.
//
// Replaces the one-party `snarkjs setup --protocol groth` (prover/package.json:34,37), whose caller knows tau, alpha
// and beta, with the usual two phases: public phase-1 powers (nobody knows tau) turned into the circuit key here,
// then any number of phase-2 contributions that re-randomise delta and that anyone can check.
//   * Lagrange bases: inverse NTTs over curve points (radix-2 DIT stages in global memory, one scalar_mul per
//     butterfly whose twiddle is not 1; the bit reversal is folded into the affine -> XYZZ load).
//   * Per-signal sums: one thread per nonzero computes coef * P[row] (no multiplication when coef = 1), then a
//     segmented sum in chunks of kSegChunk entries, repeated over the partials until each column has one point, so a
//     column of 10^5 entries costs log_32 levels instead of one serial thread.  The group law is exact: the order of
//     the additions cannot change the affine bytes.
//   * Contributions: one thread per C / H point multiplies by the single scalar delta'^-1 with 4-bit signed windows.
//   * Verification: two bucketed MSMs (zkr_msm) with shared random 128-bit scalars over the C|H section, and host
//     pairings (verify.cu).
#include "ceremony.cuh"
#include "ntt_iface.cuh"

using namespace zkr;

namespace {

constexpr uint32_t kSegChunk = 32;

// ------------------------------------------------------------------------------------------------ point NTT
// X[bitrev(k)] = P[k]: the DIT stages below then leave the transform in natural order
template <class F>
__global__ void k_pntt_load(const Affine<F>* __restrict__ in, XYZZ<F>* X, uint32_t m, int log_m) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    XYZZ<F>::from_affine(Affine<F>::load_ro(in + k)).store(X + (__brev(k) >> (32 - log_m)));
}

// One radix-2 DIT stage of the inverse transform (butterflies of span 2^s) over `blocks` vectors of m points
// stored back to back: (u, v) -> (u + w v, u - w v), w = omega_m^(-j m / 2^(s+1)).
template <class F>
__global__ void k_pntt_stage(XYZZ<F>* X, uint32_t m, int log_m, int s, uint32_t blocks, const Fr* __restrict__ tw_lo,
                             const Fr* __restrict__ tw_hi, int lb) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= blocks * (m / 2)) return;
    const uint32_t b = t >> (log_m - 1), tb = t & (m / 2 - 1);
    const uint32_t j = tb & ((1u << s) - 1);
    XYZZ<F>* x = X + (size_t)b * m;
    const uint32_t i0 = ((tb >> s) << (s + 1)) + j, i1 = i0 + (1u << s);
    XYZZ<F> u = XYZZ<F>::load(x + i0), v = XYZZ<F>::load(x + i1);
    if (j) {
        const uint32_t e = j << (log_m - 1 - s);
        const Fr w = Fr::load_ro(tw_lo + (e & ((1u << lb) - 1))) * Fr::load_ro(tw_hi + (e >> lb));
        v = scalar_mul(v, w.from_mont());
    }
    XYZZ<F> d = u;
    d.add(v.neg());
    u.add(v);
    u.store(x + i0);
    d.store(x + i1);
}

// X[i] *= 1/m
template <class F>
__global__ void k_pntt_scale(XYZZ<F>* X, size_t n, const NttRoots* roots) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    scalar_mul(XYZZ<F>::load(X + i), roots->ninv.from_mont()).store(X + i);
}

// H_k = [tau^(k+m)] - [tau^k]; infinity where tau^(k+m) is not given (k = m - 1 with 2m - 1 powers)
__global__ void k_h_from_powers(const G1Affine* __restrict__ tau, uint32_t n_tau, G1Affine* out, uint32_t m) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    G1XYZZ acc = G1XYZZ::identity();
    if (k + m < n_tau) {
        acc = G1XYZZ::from_affine(G1Affine::load_ro(tau + k + m));
        acc.madd(G1Affine::load_ro(tau + k).neg());
    }
    store_key_point(acc, out + k);
}

// ------------------------------------------------------------------------------------------------ sparse sums
// T[k] = cid-th pool coefficient (std form) * P[pidx[k]]
template <class F>
__global__ void k_terms(const XYZZ<F>* __restrict__ P, const uint32_t* __restrict__ pidx, const uint32_t* __restrict__ cid,
                        const Fr* __restrict__ pool, XYZZ<F>* T, uint32_t nnz) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    const XYZZ<F> p = XYZZ<F>::load(P + pidx[k]);
    const Fr c = Fr::load_ro(pool + cid[k]);
    bool one = c.v[0] == 1;
#pragma unroll
    for (int i = 1; i < 8; i++) one &= c.v[i] == 0;
    (one ? p : scalar_mul(p, c)).store(T + k);
}

// out[c] = sum of in[start[c] .. start[c+1])
template <class F>
__global__ void k_seg_sum(const XYZZ<F>* __restrict__ in, const uint32_t* __restrict__ start, XYZZ<F>* out, uint32_t nch) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nch) return;
    const uint32_t e = start[c + 1];
    XYZZ<F> acc = XYZZ<F>::load(in + start[c]);
#pragma unroll 1
    for (uint32_t k = start[c] + 1; k < e; k++) acc.add(XYZZ<F>::load(in + k));
    acc.store(out + c);
}

// column i holds at most one point, in[ptr[i]]; an empty column is infinity
template <class F>
__global__ void k_col_affine(const XYZZ<F>* __restrict__ in, const uint32_t* __restrict__ ptr, Affine<F>* out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    store_key_point(ptr[i + 1] > ptr[i] ? XYZZ<F>::load(in + ptr[i]) : XYZZ<F>::identity(), out + i);
}

// ------------------------------------------------------------------------------------------------ contribution
// Device copy of the contribution's secrets, std form
struct Secrets {
    Fr delta, k;                        // delta' and the Schnorr nonce
    Fr dinv;                            // delta'^-1
    Fr c, z;                            // challenge and response (public)
};

__global__ void k_delta_inverse(Secrets* s) { s->dinv = s->delta.to_mont().inverse().from_mont(); }

// ------------------------------------------------------------------------------------------------ host helpers

// ---- websnark binary key layout (binarify.ts:152-202): 10 x u32 header, fixed block, then seven sections
constexpr size_t kPkFixed = 40;                     // alfa1 | beta1 | delta1 | beta2 | delta2
constexpr size_t kPkDelta1 = kPkFixed + 128, kPkDelta2 = kPkFixed + 320, kPkPols = kPkFixed + 448;
constexpr size_t kVkDelta1 = 128, kVkDelta2 = 448, kVkIC = 576;
struct KeyLayout {
    uint32_t n, l, m, pA, pB, pPA, pPB1, pPB2, pPC, pPH;
};
bool key_layout(const void* pk, size_t len, size_t vk_len, KeyLayout* v) {
    if (len < kPkPols) return false;
    memcpy(v, pk, 40);
    const uint64_t n = v->n, l = v->l, m = v->m;
    return n >= 1 && l + 1 <= n && m >= 2 && (m & (m - 1)) == 0 && v->pA == kPkPols && v->pA <= v->pB && v->pB <= v->pPA &&
           (uint64_t)v->pPA + 64 * n == v->pPB1 && (uint64_t)v->pPB1 + 64 * n == v->pPB2 &&
           (uint64_t)v->pPB2 + 128 * n == v->pPC && (uint64_t)v->pPC + 64 * (n - l - 1) == v->pPH &&
           (uint64_t)v->pPH + 64 * m == len && vk_len == kVkIC + 64 * (l + 1);
}

// ---- setup_from_powers input checks

// CSC columns of one sum: for column i, entries [ptr[i], ptr[i+1]) of (point index, pool index)
struct Cols {
    std::vector<uint32_t> ptr, pidx, cid;
};

// d_out[i] = sum over column i of pool[cid] * P[pidx], key encoding
template <class F>
int combine(zkr_ctx* ctx, cudaStream_t st, const XYZZ<F>* d_pts, const Cols& c, const Fr* d_pool, Affine<F>* d_out) {
    const uint32_t n = (uint32_t)c.ptr.size() - 1;
    const uint32_t nnz = c.ptr[n];
    DevAllocs a;
    XYZZ<F>* T = nullptr;
    if (nnz) {
        uint32_t *d_idx, *d_cid;
        ZKR_TRY(a.upload(&d_idx, c.pidx.data(), nnz, st));
        ZKR_TRY(a.upload(&d_cid, c.cid.data(), nnz, st));
        ZKR_TRY(a.alloc(&T, sizeof(XYZZ<F>) * (size_t)nnz));
        ZKR_LAUNCH(ctx, k_terms<F>, ceil_div(nnz, 128), 128, 0, st, d_pts, d_idx, d_cid, d_pool, T, nnz);
        ZKR_CUDA(cudaStreamSynchronize(st));
        a.release(d_idx);
        a.release(d_cid);
    }
    std::vector<uint32_t> ptr = c.ptr;
    for (;;) {
        uint32_t mx = 0;
        for (uint32_t i = 0; i < n; i++) mx = std::max(mx, ptr[i + 1] - ptr[i]);
        if (mx <= 1) break;
        std::vector<uint32_t> start, next(n + 1, 0);
        for (uint32_t i = 0; i < n; i++) {
            for (uint32_t s = ptr[i]; s < ptr[i + 1]; s += kSegChunk) start.push_back(s);
            next[i + 1] = (uint32_t)start.size();
        }
        start.push_back(ptr[n]);
        const uint32_t nch = (uint32_t)start.size() - 1;
        uint32_t* d_start;
        XYZZ<F>* U;
        ZKR_TRY(a.upload(&d_start, start.data(), start.size(), st));
        ZKR_TRY(a.alloc(&U, sizeof(XYZZ<F>) * (size_t)nch));
        ZKR_LAUNCH(ctx, k_seg_sum<F>, ceil_div(nch, 128), 128, 0, st, T, d_start, U, nch);
        ZKR_CUDA(cudaStreamSynchronize(st));
        a.release(d_start);
        a.release(T);
        T = U;
        ptr.swap(next);
    }
    uint32_t* d_ptr;
    ZKR_TRY(a.upload(&d_ptr, ptr.data(), ptr.size(), st));
    ZKR_LAUNCH(ctx, k_col_affine<F>, ceil_div(n, 128), 128, 0, st, T, d_ptr, d_out, n);
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

// Inverse NTT of `blocks` vectors of m points each, in place: natural order in (after k_pntt_load), natural out.
template <class F>
int point_intt(zkr_ctx* ctx, cudaStream_t st, XYZZ<F>* X, uint32_t blocks, int log_m, const NttTables* tv) {
    const uint32_t m = 1u << log_m, nb = blocks * (m / 2);
    for (int s = 0; s < log_m; s++)
        ZKR_LAUNCH(ctx, k_pntt_stage<F>, ceil_div(nb, 128), 128, 0, st, X, m, log_m, s, blocks, tv->tw_lo_i, tv->tw_hi_i, tv->lb);
    ZKR_LAUNCH(ctx, k_pntt_scale<F>, ceil_div((size_t)blocks * m, 128), 128, 0, st, X, (size_t)blocks * m, tv->roots);
    return ZKR_OK;
}

template <class F>
int load_points(zkr_ctx* ctx, cudaStream_t st, const void* h_pts, Affine<F>* d_stage, XYZZ<F>* X, int log_m) {
    const uint32_t m = 1u << log_m;
    ZKR_CUDA(cudaMemcpyAsync(d_stage, h_pts, sizeof(Affine<F>) * (size_t)m, cudaMemcpyHostToDevice, st));
    ZKR_LAUNCH(ctx, k_pntt_load<F>, ceil_div(m, 128), 128, 0, st, d_stage, X, m, log_m);
    return ZKR_OK;
}

template <class F>
int download(cudaStream_t st, void* h, const Affine<F>* d, size_t count) {
    if (count) ZKR_CUDA(cudaMemcpyAsync(h, d, sizeof(Affine<F>) * count, cudaMemcpyDeviceToHost, st));
    return ZKR_OK;
}

int check_r1cs(const zkr_r1cs_csc* r) {
    const uint32_t n = r->n_vars, m = r->domain_size;
    if (!r->pool || !r->n_pool) {
        set_error("zkr_setup_from_powers: empty coefficient pool");
        return ZKR_E_INVALID;
    }
    for (uint32_t i = 0; i < r->n_pool; i++)
        if (!lt_r((const uint8_t*)r->pool + 32 * (size_t)i)) {
            set_error("zkr_setup_from_powers: pool[%u] is >= r", i);
            return ZKR_E_INVALID;
        }
    const uint32_t* hp[3][3] = {{r->ptr_a, r->row_a, r->cid_a}, {r->ptr_b, r->row_b, r->cid_b}, {r->ptr_c, r->row_c, r->cid_c}};
    for (int k = 0; k < 3; k++) {
        const uint32_t *ptr = hp[k][0], *row = hp[k][1], *cid = hp[k][2];
        bool ok = ptr && ptr[0] == 0 && (ptr[n] == 0 || (row && cid));
        for (uint32_t i = 0; ok && i < n; i++) ok = ptr[i] <= ptr[i + 1];
        for (uint32_t e = 0; ok && e < ptr[n]; e++) ok = row[e] < m && cid[e] < r->n_pool;
        if (!ok) {
            set_error("zkr_setup_from_powers: matrix %c: column pointers not monotone, a row >= domain_size or a pool index "
                      ">= n_pool", "ABC"[k]);
            return ZKR_E_INVALID;
        }
    }
    return ZKR_OK;
}

Cols columns(const uint32_t* ptr, const uint32_t* row, const uint32_t* cid, uint32_t n, uint32_t offset) {
    Cols c;
    c.ptr.assign(ptr, ptr + n + 1);
    c.pidx.resize(ptr[n]);
    for (uint32_t e = 0; e < ptr[n]; e++) c.pidx[e] = row[e] + offset;
    c.cid.assign(cid, cid + ptr[n]);
    return c;
}

}  // namespace

extern "C" int zkr_setup_from_powers(zkr_ctx* ctx, const zkr_r1cs_csc* r, const zkr_powers* pw, void* out_a, void* out_b1,
                                     void* out_b2, void* out_c, void* out_h, void* out_vk) {
    if (!ctx || !r || !pw || !out_a || !out_b1 || !out_b2 || !out_c || !out_h || !out_vk) return ZKR_E_INVALID;
    const uint32_t n = r->n_vars, l = r->n_public, m = r->domain_size;
    if (n == 0 || l + 1 > n || (m & (m - 1)) || m < 2 || m > (1u << 27) || r->n_constraints + l + 1 > m) {
        set_error("zkr_setup_from_powers: inconsistent R1CS shape");
        return ZKR_E_INVALID;
    }
    ZKR_TRY(check_r1cs(r));
    const uint32_t n_tau = std::min(pw->n_tau_g1, 2 * m);      // tau^(2m-1), when given, makes H_(m-1)
    ZKR_TRY(check_section("zkr_setup_from_powers", "tau_g1", 1, pw->tau_g1, pw->n_tau_g1, 2 * m - 1, n_tau));
    ZKR_TRY(check_section("zkr_setup_from_powers", "tau_g2", 2, pw->tau_g2, pw->n_tau_g2, m, m));
    ZKR_TRY(check_section("zkr_setup_from_powers", "alpha_tau_g1", 1, pw->alpha_tau_g1, pw->n_alpha_tau_g1, m, m));
    ZKR_TRY(check_section("zkr_setup_from_powers", "beta_tau_g1", 1, pw->beta_tau_g1, pw->n_beta_tau_g1, m, m));
    ZKR_TRY(check_section("zkr_setup_from_powers", "beta_g2", 2, pw->beta_g2, 1, 1, 1));

    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    int log_m = 0;
    while ((1u << log_m) < m) log_m++;
    NttTables* tabs;
    ZKR_TRY(ntt_get_tables(ctx, log_m, &tabs));
    const NttTables* tv = tabs;

    // P1 = [L | alpha L | beta L] (G1), P2 = L (G2), XYZZ
    DevAllocs a;
    G1Affine *d_tau, *d_stage1, *d_out1;
    G2Affine *d_stage2, *d_out2;
    G1XYZZ* P1;
    G2XYZZ* P2;
    Fr* d_pool;
    ZKR_TRY(a.alloc(&d_stage1, sizeof(G1Affine) * (size_t)m));
    ZKR_TRY(a.alloc(&d_stage2, sizeof(G2Affine) * (size_t)m));
    ZKR_TRY(a.alloc(&d_out1, sizeof(G1Affine) * (size_t)std::max(n, m)));
    ZKR_TRY(a.alloc(&d_out2, sizeof(G2Affine) * (size_t)n));
    ZKR_TRY(a.alloc(&P1, sizeof(G1XYZZ) * 3 * (size_t)m));
    ZKR_TRY(a.alloc(&P2, sizeof(G2XYZZ) * (size_t)m));
    ZKR_TRY(a.upload(&d_pool, r->pool, r->n_pool, st));
    ZKR_TRY(a.upload(&d_tau, pw->tau_g1, n_tau, st));

    // H straight from the powers
    ZKR_LAUNCH(ctx, k_h_from_powers, ceil_div(m, 128), 128, 0, st, d_tau, n_tau, d_out1, m);
    ZKR_TRY(download(st, out_h, d_out1, m));
    ZKR_CUDA(cudaStreamSynchronize(st));

    // Lagrange bases
    ZKR_LAUNCH(ctx, k_pntt_load<Fq>, ceil_div(m, 128), 128, 0, st, d_tau, P1, m, log_m);
    ZKR_TRY(load_points<Fq>(ctx, st, pw->alpha_tau_g1, d_stage1, P1 + m, log_m));
    ZKR_TRY(load_points<Fq>(ctx, st, pw->beta_tau_g1, d_stage1, P1 + 2 * (size_t)m, log_m));
    ZKR_TRY(load_points<Fq2>(ctx, st, pw->tau_g2, d_stage2, P2, log_m));
    ZKR_TRY(point_intt<Fq>(ctx, st, P1, 3, log_m, tv));
    ZKR_TRY(point_intt<Fq2>(ctx, st, P2, 1, log_m, tv));

    // per-signal sums
    const Cols ca = columns(r->ptr_a, r->row_a, r->cid_a, n, 0);
    const Cols cb = columns(r->ptr_b, r->row_b, r->cid_b, n, 0);
    ZKR_TRY(combine<Fq>(ctx, st, P1, ca, d_pool, d_out1));
    ZKR_TRY(download(st, out_a, d_out1, n));
    ZKR_CUDA(cudaStreamSynchronize(st));
    ZKR_TRY(combine<Fq>(ctx, st, P1, cb, d_pool, d_out1));
    ZKR_TRY(download(st, out_b1, d_out1, n));
    ZKR_TRY(combine<Fq2>(ctx, st, P2, cb, d_pool, d_out2));
    ZKR_TRY(download(st, out_b2, d_out2, n));
    // IC / C: a [beta L] + b [alpha L] + c [L], the three matrices' entries of a column back to back
    Cols cc;
    cc.ptr.assign(n + 1, 0);
    const uint32_t* hp[3][3] = {{r->ptr_a, r->row_a, r->cid_a}, {r->ptr_b, r->row_b, r->cid_b}, {r->ptr_c, r->row_c, r->cid_c}};
    const uint32_t block[3] = {2 * m, m, 0};
    for (uint32_t i = 0; i < n; i++) {
        for (int k = 0; k < 3; k++)
            for (uint32_t e = hp[k][0][i]; e < hp[k][0][i + 1]; e++) {
                cc.pidx.push_back(hp[k][1][e] + block[k]);
                cc.cid.push_back(hp[k][2][e]);
            }
        cc.ptr[i + 1] = (uint32_t)cc.pidx.size();
    }
    ZKR_TRY(combine<Fq>(ctx, st, P1, cc, d_pool, d_out1));
    char* vk = (char*)out_vk;
    ZKR_TRY(download(st, vk + kVkIC, d_out1, l + 1));
    ZKR_TRY(download(st, out_c, d_out1 + l + 1, n - l - 1));
    // vk: alfa1 | beta1 | delta1 = G1 | beta2 | gamma2 = G2 | delta2 = G2
    uint8_t gen[192];
    ZKR_TRY(generators(ctx, st, gen));
    memcpy(vk, pw->alpha_tau_g1, 64);
    memcpy(vk + 64, pw->beta_tau_g1, 64);
    memcpy(vk + 128, gen, 64);
    memcpy(vk + 192, pw->beta_g2, 128);
    memcpy(vk + 320, gen + 64, 128);
    memcpy(vk + 448, gen + 64, 128);
    return ZKR_OK;
}

extern "C" int zkr_setup_contribute(zkr_ctx* ctx, const void* pk, size_t pk_len, const void* vk, size_t vk_len,
                                    const void* delta32, void* out_pk, void* out_vk, void* out_record) {
    if (!ctx || !pk || !vk || !out_pk || !out_vk || !out_record) return ZKR_E_INVALID;
    KeyLayout L;
    if (!key_layout(pk, pk_len, vk_len, &L)) {
        set_error("zkr_setup_contribute: proving key / vk layout inconsistent (len %zu, vk %zu)", pk_len, vk_len);
        return ZKR_E_INVALID;
    }
    const uint8_t* p = (const uint8_t*)pk;
    const uint8_t* v = (const uint8_t*)vk;
    if (memcmp(p + kPkDelta1, v + kVkDelta1, 64) || memcmp(p + kPkDelta2, v + kVkDelta2, 128)) {
        set_error("zkr_setup_contribute: the key header and the vk disagree on delta");
        return ZKR_E_INVALID;
    }
    if (host_point_check(1, p + kPkDelta1, false) != PT_OK || host_point_check(2, p + kPkDelta2, true) != PT_OK) {
        set_error("zkr_setup_contribute: delta1 / delta2 is not a valid point");
        return ZKR_E_INVALID;
    }
    if (delta32 && (is_zero32((const uint8_t*)delta32) || !lt_r((const uint8_t*)delta32))) {
        set_error("zkr_setup_contribute: delta must be in [1, r)");
        return ZKR_E_INVALID;
    }
    // host secrets: delta' then k, both nonzero
    HostSecret<64> sec;
    if (delta32) memcpy(sec.b, delta32, 32);
    else ZKR_TRY(draw_nonzero(sec.b));
    ZKR_TRY(draw_nonzero(sec.b + 32));

    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    const size_t nch = (size_t)(L.n - L.l - 1) + L.m;          // C | H, contiguous
    DevAllocs a;
    Secrets* d_sec;
    G1Affine *d_ch, *d_g1;
    G2Affine* d_g2;
    ZKR_TRY(a.alloc_secret(&d_sec, sizeof(Secrets), st));
    ZKR_CUDA(cudaMemcpyAsync(d_sec, sec.b, 64, cudaMemcpyHostToDevice, st));      // delta, k
    ZKR_TRY(a.upload(&d_ch, p + L.pPC, nch, st));
    ZKR_TRY(a.alloc(&d_g1, 128));
    ZKR_CUDA(cudaMemcpyAsync(d_g1, p + kPkDelta1, 64, cudaMemcpyHostToDevice, st));
    ZKR_CUDA(cudaMemcpyAsync(d_g1 + 1, p + kPkDelta1, 64, cudaMemcpyHostToDevice, st));
    ZKR_TRY(a.upload(&d_g2, p + kPkDelta2, 1, st));
    // C | H by delta'^-1; delta1, delta2 by delta'; R = k delta1_old
    ZKR_LAUNCH(ctx, k_delta_inverse, 1, 1, 0, st, d_sec);
    ZKR_LAUNCH(ctx, k_scale_points<Fq>, ceil_div(nch, 128), 128, 0, st, d_ch, nch, nullptr, nullptr, &d_sec->dinv);
    ZKR_LAUNCH(ctx, k_scale_points<Fq>, 1, 1, 0, st, d_g1, (size_t)1, nullptr, nullptr, &d_sec->delta);
    ZKR_LAUNCH(ctx, k_scale_points<Fq>, 1, 1, 0, st, d_g1 + 1, (size_t)1, nullptr, nullptr, &d_sec->k);
    ZKR_LAUNCH(ctx, k_scale_points<Fq2>, 1, 1, 0, st, d_g2, (size_t)1, nullptr, nullptr, &d_sec->delta);
    uint8_t small[64 * 2 + 128];                               // delta1_new | R | delta2_new
    ZKR_CUDA(cudaMemcpyAsync((uint8_t*)out_pk + L.pPC, d_ch, 64 * nch, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaMemcpyAsync(small, d_g1, 128, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaMemcpyAsync(small + 128, d_g2, 128, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    uint8_t c[32];
    challenge("zkr-phase2-delta", p + kPkDelta1, small, small + 64, c);
    ZKR_CUDA(cudaMemcpyAsync(&d_sec->c, c, 32, cudaMemcpyHostToDevice, st));
    ZKR_LAUNCH(ctx, k_schnorr_z, 1, 1, 0, st, &d_sec->delta, &d_sec->k, &d_sec->c, &d_sec->z, 1);
    ZKR_CUDA(cudaMemcpyAsync((uint8_t*)out_record + 64, &d_sec->z, 32, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));

    uint8_t* op = (uint8_t*)out_pk;
    uint8_t* ov = (uint8_t*)out_vk;
    memcpy(op, p, L.pPC);
    memcpy(ov, v, vk_len);
    memcpy(op + kPkDelta1, small, 64);
    memcpy(ov + kVkDelta1, small, 64);
    memcpy(op + kPkDelta2, small + 128, 128);
    memcpy(ov + kVkDelta2, small + 128, 128);
    memcpy(out_record, small + 64, 64);
    return ZKR_OK;
}

extern "C" int zkr_setup_verify_contribution(zkr_ctx* ctx, const void* old_pk, const void* old_vk, const void* new_pk,
                                             const void* new_vk, size_t pk_len, size_t vk_len, const void* record,
                                             int* valid) {
    if (!ctx || !old_pk || !old_vk || !new_pk || !new_vk || !record || !valid) return ZKR_E_INVALID;
    *valid = 0;
    KeyLayout L;
    if (!key_layout(old_pk, pk_len, vk_len, &L)) {
        set_error("zkr_setup_verify_contribution: proving key / vk layout inconsistent (len %zu, vk %zu)", pk_len, vk_len);
        return ZKR_E_INVALID;
    }
    const uint8_t *po = (const uint8_t*)old_pk, *pn = (const uint8_t*)new_pk;
    const uint8_t *vo = (const uint8_t*)old_vk, *vn = (const uint8_t*)new_vk;
    const uint8_t* R = (const uint8_t*)record;
    // every byte outside delta1, delta2, C and H
    const size_t pk_same[3][2] = {{0, kPkDelta1}, {kPkDelta1 + 64, kPkDelta2}, {kPkDelta2 + 128, L.pPC}};
    const size_t vk_same[3][2] = {{0, kVkDelta1}, {kVkDelta1 + 64, kVkDelta2}, {kVkDelta2 + 128, vk_len}};
    for (int i = 0; i < 3; i++)
        if (memcmp(po + pk_same[i][0], pn + pk_same[i][0], pk_same[i][1] - pk_same[i][0]) ||
            memcmp(vo + vk_same[i][0], vn + vk_same[i][0], vk_same[i][1] - vk_same[i][0]))
            return ZKR_OK;
    const uint8_t* keys[2][2] = {{po, vo}, {pn, vn}};
    for (auto& k : keys) {
        if (memcmp(k[0] + kPkDelta1, k[1] + kVkDelta1, 64) || memcmp(k[0] + kPkDelta2, k[1] + kVkDelta2, 128)) return ZKR_OK;
        if (host_point_check(1, k[0] + kPkDelta1, false) != PT_OK || host_point_check(2, k[0] + kPkDelta2, true) != PT_OK)
            return ZKR_OK;
    }
    if (host_point_check(1, R, false) != PT_OK || !lt_r(R + 64)) return ZKR_OK;

    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    // e(delta1_new, G2) = e(G1, delta2_new)
    uint8_t gen[192];
    ZKR_TRY(generators(ctx, st, gen));
    {
        const void* P[2] = {pn + kPkDelta1, gen};
        const void* Q[2] = {gen + 64, pn + kPkDelta2};
        const bool neg[2] = {true, false};
        if (!host_pairing_is_one(P, neg, Q, 2)) return ZKR_OK;
    }
    // z delta1_old = R + c delta1_new
    bool ok;
    ZKR_TRY(schnorr_holds(ctx, st, "zkr-phase2-delta", po + kPkDelta1, pn + kPkDelta1, R, R + 64, &ok));
    if (!ok) return ZKR_OK;
    // every new C / H point in range and on the curve (the MSM formulas do not see the curve constant), and an
    // infinity written as an honest contribution writes it, (0, R mod q): R mod q is the generator's x
    const size_t nch = (size_t)(L.n - L.l - 1) + L.m;
    int code;
    if (first_bad_point(1, pn + L.pPC, nch, gen, &code) < nch) return ZKR_OK;
    // e(X_new, delta2_new) = e(X_old, delta2_old), X = sum rho_i C_i + sum sigma_k H_k, 128-bit rho / sigma
    std::vector<uint8_t> sc(32 * nch, 0);
    {
        std::vector<uint8_t> rnd(16 * nch);
        ZKR_TRY(os_random(rnd.data(), rnd.size()));
        for (size_t i = 0; i < nch; i++) memcpy(&sc[32 * i], &rnd[16 * i], 16);
    }
    uint8_t X[2][64];
    const uint8_t* src[2] = {po, pn};
    for (int s = 0; s < 2; s++) {
        zkr_bases* b = nullptr;
        ZKR_TRY(zkr_bases_load(ctx, 1, src[s] + L.pPC, nch, 0, &b));
        uint8_t xs[64];
        const int rc = zkr_msm(ctx, b, sc.data(), nch, 0, xs);
        zkr_bases_free(b);
        ZKR_TRY(rc);
        if (!host_g1_std_to_mont(xs, X[s])) {
            set_error("zkr_setup_verify_contribution: MSM result out of range");
            return ZKR_E_CUDA;
        }
    }
    const void* P[2] = {X[1], X[0]};
    const void* Q[2] = {pn + kPkDelta2, po + kPkDelta2};
    const bool neg[2] = {false, true};
    *valid = host_pairing_is_one(P, neg, Q, 2) ? 1 : 0;
    return ZKR_OK;
}
