// Synthetic Groth16 trusted setup on the GPU (C-ABI: zkr_synth_setup).
//
// Stands where the reference runs `snarkjs setup --protocol groth`
// (/root/reference/prover/package.json:34,37) -- for SYNTHETIC circuits only: the toxic waste
// (tau, alpha, beta, gamma, delta) is an INPUT, so keys made here are test / benchmark keys.
// The reference commits no proving key (prover/.gitignore: build/), and circom cannot run in this
// environment, so benchmarks need keys of the rollup's shape at 2^17..2^22 constraints; a CPU setup
// at that size takes hours in Python, the GPU does it in well under a second.
// Math: SURVEY.md B.5 (oracle: oracle/groth16.py setup()).  Output point encoding follows
// binarifyProvingKey (/root/reference/operator/src/utils/binarify.ts:92-102): affine, Fq-M,
// infinity written as (0, R mod q) because snarkjs's affine zero is [0, 1, 0].
#include "ec.cuh"
#include "msm_iface.cuh"
#include "ntt_iface.cuh"

using namespace zkr;

namespace {

constexpr int kFbWin = 32;    // 32 windows of 8 bits

// base[w] = 2^(8w) G
template <class F>
__global__ void k_fb_base(Affine<F>* base) {
    XYZZ<F> p = XYZZ<F>::from_affine(generator<F>());
    for (int w = 0; w < kFbWin; w++) {
        p.to_affine().store(base + w);
#pragma unroll 1
        for (int d = 0; d < 8; d++) p = p.dbl();
    }
}

// table[w][d] = d * base[w], d = 1..255
template <class F>
__global__ void k_fb_table(const Affine<F>* base, Affine<F>* table) {
    const int w = blockIdx.x, d = threadIdx.x;
    if (d == 0) return;
    XYZZ<F> p = XYZZ<F>::from_affine(Affine<F>::load(base + w));
    Fr k = Fr::zero();
    k.v[0] = d;
    scalar_mul(p, k).to_affine().store(table + w * 256 + d);
}

// out[i] = scalars[i] * G  (affine Montgomery; infinity -> (0, one))
template <class F>
__global__ void k_fb_mul(const Fr* __restrict__ scalars, const Affine<F>* __restrict__ table, Affine<F>* out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr k = Fr::load(scalars + i);
    XYZZ<F> acc = XYZZ<F>::identity();
#pragma unroll 1
    for (int w = 0; w < kFbWin; w++) {
        const uint32_t d = (k.v[w >> 2] >> ((w & 3) * 8)) & 0xff;
        if (d) acc.madd(Affine<F>::load_ro(table + w * 256 + d));
    }
    Affine<F> a = acc.to_affine();
    if (acc.is_inf()) a.y = F::one();
    a.store(out + i);
}

__device__ __forceinline__ Fr pow_u64(Fr base, unsigned long long e) {
    Fr acc = Fr::one();
    while (e) {
        if (e & 1) acc = acc * base;
        base = base.sqr();
        e >>= 1;
    }
    return acc;
}

struct Toxic {
    Fr tau, alpha, beta, gamma, delta;   // Montgomery
    Fr zt;                                // tau^m - 1
    Fr dinv, ginv, minv;
};

__global__ void k_toxic(const Fr* in_std, Toxic* out, uint32_t m) {
    Toxic t;
    t.tau = Fr::load(in_std).to_mont();
    t.alpha = Fr::load(in_std + 1).to_mont();
    t.beta = Fr::load(in_std + 2).to_mont();
    t.gamma = Fr::load(in_std + 3).to_mont();
    t.delta = Fr::load(in_std + 4).to_mont();
    t.zt = pow_u64(t.tau, m) - Fr::one();
    t.dinv = t.delta.inverse();
    t.ginv = t.gamma.inverse();
    Fr mm = Fr::zero();
    mm.v[0] = m;
    t.minv = mm.to_mont().inverse();
    *out = t;
}

// L_c(tau) = omega^c (tau^m - 1) / (m (tau - omega^c)),  Montgomery form
__global__ void k_lagrange(Fr* L, uint32_t m, const Toxic* tx, const Fr* tw_lo, const Fr* tw_hi, int lb) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    Fr wc = Fr::load_ro(tw_lo + (c & ((1u << lb) - 1))) * Fr::load_ro(tw_hi + (c >> lb));
    Fr den = (tx->tau - wc).inverse();
    (wc * tx->zt * tx->minv * den).store(L + c);
}

__global__ void k_to_mont(Fr* x, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) Fr::load(x + i).to_mont().store(x + i);
}

// out[i] = sum_k pool[cid[k]] * L[row[k]] over column i
__global__ void k_col_eval(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ row,
                           const uint32_t* __restrict__ cid, const Fr* __restrict__ pool, const Fr* __restrict__ L,
                           Fr* out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = Fr::zero();
    const uint32_t e = ptr[i + 1];
    for (uint32_t k = ptr[i]; k < e; k++) acc = acc + Fr::load_ro(pool + cid[k]) * Fr::load_ro(L + row[k]);
    acc.store(out + i);
}

// standard-form scalars for the fixed-base multiplications
__global__ void k_setup_scalars(const Fr* at, const Fr* bt, const Fr* ct, const Toxic* tx, uint32_t n, uint32_t l,
                                uint32_t m, Fr* sA, Fr* sB, Fr* sC, Fr* sIC, Fr* sH, Fr* sVK) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t top = n > m ? n : m;
    if (i >= top) return;
    if (i < n) {
        Fr a = Fr::load(at + i), b = Fr::load(bt + i), c = Fr::load(ct + i);
        a.from_mont().store(sA + i);
        b.from_mont().store(sB + i);
        Fr k = tx->beta * a + tx->alpha * b + c;
        if (i <= l) (k * tx->ginv).from_mont().store(sIC + i);
        else (k * tx->dinv).from_mont().store(sC + (i - l - 1));
    }
    if (i < m) (pow_u64(tx->tau, i) * tx->zt * tx->dinv).from_mont().store(sH + i);
    if (i == 0) {
        tx->alpha.from_mont().store(sVK);
        tx->beta.from_mont().store(sVK + 1);
        tx->delta.from_mont().store(sVK + 2);
        tx->gamma.from_mont().store(sVK + 3);
    }
}

template <class F>
int fixed_base(zkr_ctx* ctx, cudaStream_t st, Affine<F>* table, const Fr* d_scalars, uint32_t n, void* h_out) {
    if (n == 0) return ZKR_OK;
    DevAllocs a;
    Affine<F>* d_out;
    ZKR_TRY(a.alloc(&d_out, sizeof(Affine<F>) * (size_t)n));
    ZKR_LAUNCH(ctx, k_fb_mul<F>, ceil_div(n, 64), 64, 0, st, d_scalars, table, d_out, n);
    ZKR_CUDA(cudaMemcpyAsync(h_out, d_out, sizeof(Affine<F>) * (size_t)n, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

// *table = the fixed-base table of the generator, owned by `owner`
template <class F>
int build_table(zkr_ctx* ctx, cudaStream_t st, DevAllocs& owner, Affine<F>** table) {
    DevAllocs a;
    Affine<F>* base;
    ZKR_TRY(a.alloc(&base, sizeof(Affine<F>) * kFbWin));
    ZKR_TRY(owner.alloc(table, sizeof(Affine<F>) * kFbWin * 256));
    ZKR_CUDA(cudaMemsetAsync(*table, 0, sizeof(Affine<F>) * kFbWin * 256, st));
    ZKR_LAUNCH(ctx, k_fb_base<F>, 1, 1, 0, st, base);
    ZKR_LAUNCH(ctx, k_fb_table<F>, kFbWin, 256, 0, st, (const Affine<F>*)base, *table);
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

}  // namespace

extern "C" int zkr_synth_setup(zkr_ctx* ctx, const zkr_r1cs_csc* r, const void* toxic, void* out_a, void* out_b1,
                               void* out_b2, void* out_c, void* out_h, void* out_vk) {
    if (!ctx || !r || !toxic || !out_a || !out_b1 || !out_b2 || !out_c || !out_h || !out_vk) return ZKR_E_INVALID;
    const uint32_t n = r->n_vars, l = r->n_public, m = r->domain_size;
    if (n == 0 || l + 1 > n || (m & (m - 1)) || m < 2 || r->n_constraints + l + 1 > m) {
        set_error("zkr_synth_setup: inconsistent R1CS shape");
        return ZKR_E_INVALID;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    int log_m = 0;
    while ((1u << log_m) < m) log_m++;
    NttTables* tabs;
    ZKR_TRY(ntt_get_tables(ctx, log_m, &tabs));
    const NttTables* tv = tabs;

    DevAllocs a;
    Fr *d_tox_in, *d_pool, *d_L, *d_at, *d_bt, *d_ct, *sA, *sB, *sC, *sIC, *sH, *sVK;
    Toxic* d_tox;
    ZKR_TRY(a.upload(&d_tox_in, toxic, 5, st));
    ZKR_TRY(a.alloc(&d_tox, sizeof(Toxic)));
    ZKR_TRY(a.upload(&d_pool, r->pool, r->n_pool, st));
    ZKR_TRY(a.alloc(&d_L, 32 * (size_t)m));
    ZKR_TRY(a.alloc(&d_at, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&d_bt, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&d_ct, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&sA, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&sB, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&sC, 32 * (size_t)n));
    ZKR_TRY(a.alloc(&sIC, 32 * (size_t)(l + 1)));
    ZKR_TRY(a.alloc(&sH, 32 * (size_t)m));
    ZKR_TRY(a.alloc(&sVK, 32 * 4));
    ZKR_LAUNCH(ctx, k_to_mont, ceil_div(r->n_pool, 128), 128, 0, st, d_pool, r->n_pool);
    ZKR_LAUNCH(ctx, k_toxic, 1, 1, 0, st, d_tox_in, d_tox, m);
    ZKR_LAUNCH(ctx, k_lagrange, ceil_div(m, 128), 128, 0, st, d_L, m, d_tox, tv->tw_lo_f, tv->tw_hi_f, tv->lb);
    const uint32_t* hp[3][3] = {{r->ptr_a, r->row_a, r->cid_a}, {r->ptr_b, r->row_b, r->cid_b}, {r->ptr_c, r->row_c, r->cid_c}};
    Fr* outs[3] = {d_at, d_bt, d_ct};
    for (int k = 0; k < 3; k++) {
        const uint32_t nnz = hp[k][0][n];
        DevAllocs cols;
        uint32_t *dp, *dr, *dc;
        ZKR_TRY(cols.upload(&dp, hp[k][0], (size_t)n + 1, st));
        ZKR_TRY(cols.upload(&dr, hp[k][1], nnz, st));
        ZKR_TRY(cols.upload(&dc, hp[k][2], nnz, st));
        ZKR_LAUNCH(ctx, k_col_eval, ceil_div(n, 128), 128, 0, st, dp, dr, dc, d_pool, d_L, outs[k], n);
        ZKR_CUDA(cudaStreamSynchronize(st));
    }
    const uint32_t top = n > m ? n : m;
    ZKR_LAUNCH(ctx, k_setup_scalars, ceil_div(top, 128), 128, 0, st, d_at, d_bt, d_ct, d_tox, n, l, m, sA, sB, sC, sIC,
               sH, sVK);
    G1Affine* t1;
    G2Affine* t2;
    ZKR_TRY(build_table<Fq>(ctx, st, a, &t1));
    ZKR_TRY(build_table<Fq2>(ctx, st, a, &t2));
    char* vk = (char*)out_vk;
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sA, n, out_a));
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sB, n, out_b1));
    ZKR_TRY(fixed_base<Fq2>(ctx, st, t2, sB, n, out_b2));
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sC, n - l - 1, out_c));
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sH, m, out_h));
    // vk: alfa1 | beta1 | delta1 | beta2 | gamma2 | delta2 | IC      (sVK = alpha, beta, delta, gamma)
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sVK, 3, vk));
    ZKR_TRY(fixed_base<Fq2>(ctx, st, t2, sVK + 1, 1, vk + 192));          // beta2
    ZKR_TRY(fixed_base<Fq2>(ctx, st, t2, sVK + 3, 1, vk + 192 + 128));    // gamma2
    ZKR_TRY(fixed_base<Fq2>(ctx, st, t2, sVK + 2, 1, vk + 192 + 256));    // delta2
    ZKR_TRY(fixed_base<Fq>(ctx, st, t1, sIC, l + 1, vk + 192 + 384));
    return ZKR_OK;
}

// points[i] = scalars[i] * G  (G1 or G2 generator), affine Fq-M, binarify encoding; host buffers.
extern "C" int zkr_synth_points(zkr_ctx* ctx, int group, const void* scalars, size_t n, void* out_points) {
    if (!ctx || !scalars || !out_points || (group != 1 && group != 2) || n == 0 || n > 0xffffffffull) return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->s[0];
    DevAllocs a;
    Fr* d_sc;
    ZKR_TRY(a.upload(&d_sc, scalars, n, st));
    if (group == 1) {
        G1Affine* t;
        ZKR_TRY(build_table<Fq>(ctx, st, a, &t));
        return fixed_base<Fq>(ctx, st, t, d_sc, (uint32_t)n, out_points);
    }
    G2Affine* t;
    ZKR_TRY(build_table<Fq2>(ctx, st, a, &t));
    return fixed_base<Fq2>(ctx, st, t, d_sc, (uint32_t)n, out_points);
}
