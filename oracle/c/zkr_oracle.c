/* zkr_oracle.c -- CPU restatement of the Groth16 prove path of kendricktan/simple-zk-rollups.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path may link or call this file: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs use it, as the checker
 * and as the CPU baseline.  The product is simple_zk_rollups_b200/csrc (CUDA) behind include/zkr.h.
 *
 * PARITY UNPINNED: the reference's prover arithmetic lives in un-vendored npm packages
 * (websnark@0.0.5, snarkjs@0.1.20; pins: /root/reference/operator/yarn.lock:5674,6750) and the reference
 * commits no golden proof.  This file restates the published algorithm of
 *   websnark src/groth16.js groth16GenProof  (call site /root/reference/operator/src/snarks/common.ts:29)
 *     - input layouts: /root/reference/operator/src/utils/binarify.ts:10-48 (witness), :50-207 (proving key)
 *     - calcH: A, B on the 2m domain (even slots given, odd slots via iNTT_m + shifted NTT_m),
 *       pointwise multiply, iNTT_2m, upper half                               (SURVEY.md 3.2, B.4 ii)
 *     - 4 G1 multiexps + 1 G2 multiexp, blinding, affine output               (SURVEY.md B.2)
 *   snarkjs src/prover_groth.js genProof: per-point double-and-add (msm mode 0) and polfield.js
 *     recursive radix-2 FFT with omega_k = 5^((r-1)/2^k)                      (SURVEY.md 3.3)
 * and is cross-checked bit for bit against oracle/groth16.py (tests/test_oracle_c.py).
 * There is no compilable reference source under /root/reference (TypeScript / circom / Solidity only),
 * so no oracle/_ref is built; bench.py's reference arm times THIS port and says kind = "port".
 */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef unsigned __int128 u128;
typedef struct { uint64_t v[4]; } fe;
typedef struct { uint64_t p[4]; uint64_t inv; fe one, r2; } field_t;

static const field_t FQ = {
    {0x3c208c16d87cfd47ull, 0x97816a916871ca8dull, 0xb85045b68181585dull, 0x30644e72e131a029ull},
    0x87d20782e4866389ull,
    {{0xd35d438dc58f0d9dull, 0x0a78eb28f5c70b3dull, 0x666ea36f7879462cull, 0x0e0a77c19a07df2full}},
    {{0xf32cfc5b538afa89ull, 0xb5e71911d44501fbull, 0x47ab1eff0a417ff6ull, 0x06d89f71cab8351full}}};
static const field_t FR = {
    {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull},
    0xc2e1f593efffffffull,
    {{0xac96341c4ffffffbull, 0x36fc76959f60cd29ull, 0x666ea36f7879462eull, 0x0e0a77c19a07df2full}},
    {{0x1bb8e645ae216da7ull, 0x53fe3ab1e35c59e3ull, 0x8c49833d53bb8085ull, 0x0216d0b17f4e44a5ull}}};

static inline int fe_is_zero(const fe* a) { return (a->v[0] | a->v[1] | a->v[2] | a->v[3]) == 0; }
static inline int fe_eq(const fe* a, const fe* b) {
    return ((a->v[0] ^ b->v[0]) | (a->v[1] ^ b->v[1]) | (a->v[2] ^ b->v[2]) | (a->v[3] ^ b->v[3])) == 0;
}
static inline int fe_geq_p(const uint64_t* t, const field_t* F) {
    for (int i = 3; i >= 0; i--) {
        if (t[i] > F->p[i]) return 1;
        if (t[i] < F->p[i]) return 0;
    }
    return 1;
}
static inline void fe_sub_p(uint64_t* t, const field_t* F) {
    u128 b = 0;
    for (int i = 0; i < 4; i++) {
        u128 d = (u128)t[i] - F->p[i] - (uint64_t)b;
        t[i] = (uint64_t)d;
        b = (d >> 64) & 1;
    }
}
static inline void fe_add(fe* r, const fe* a, const fe* b, const field_t* F) {
    u128 c = 0;
    uint64_t t[4];
    for (int i = 0; i < 4; i++) { c += (u128)a->v[i] + b->v[i]; t[i] = (uint64_t)c; c >>= 64; }
    if (fe_geq_p(t, F)) fe_sub_p(t, F);
    memcpy(r->v, t, 32);
}
static inline void fe_sub(fe* r, const fe* a, const fe* b, const field_t* F) {
    u128 bw = 0;
    uint64_t t[4];
    for (int i = 0; i < 4; i++) {
        u128 d = (u128)a->v[i] - b->v[i] - (uint64_t)bw;
        t[i] = (uint64_t)d;
        bw = (d >> 64) & 1;
    }
    if (bw) {
        u128 c = 0;
        for (int i = 0; i < 4; i++) { c += (u128)t[i] + F->p[i]; t[i] = (uint64_t)c; c >>= 64; }
    }
    memcpy(r->v, t, 32);
}
static inline void fe_neg(fe* r, const fe* a, const field_t* F) {
    fe z = {{0, 0, 0, 0}};
    if (fe_is_zero(a)) *r = *a; else fe_sub(r, &z, a, F);
}
/* Montgomery product a*b/2^256 mod p (4x4 CIOS) */
static inline void fe_mul(fe* r, const fe* a, const fe* b, const field_t* F) {
    uint64_t t[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 4; i++) {
        u128 c = 0;
        for (int j = 0; j < 4; j++) { c += (u128)a->v[j] * b->v[i] + t[j]; t[j] = (uint64_t)c; c >>= 64; }
        c += t[4]; t[4] = (uint64_t)c; t[5] = (uint64_t)(c >> 64);
        uint64_t m = t[0] * F->inv;
        c = (u128)m * F->p[0] + t[0]; c >>= 64;
        for (int j = 1; j < 4; j++) { c += (u128)m * F->p[j] + t[j]; t[j - 1] = (uint64_t)c; c >>= 64; }
        c += t[4]; t[3] = (uint64_t)c; t[4] = t[5] + (uint64_t)(c >> 64);
    }
    if (t[4] || fe_geq_p(t, F)) fe_sub_p(t, F);
    memcpy(r->v, t, 32);
}
static inline void fe_sqr(fe* r, const fe* a, const field_t* F) { fe_mul(r, a, a, F); }
static void fe_pow(fe* r, const fe* a, const uint64_t e[4], const field_t* F) {
    fe acc = F->one, base = *a;
    for (int i = 0; i < 256; i++) {
        if ((e[i >> 6] >> (i & 63)) & 1) fe_mul(&acc, &acc, &base, F);
        fe_sqr(&base, &base, F);
    }
    *r = acc;
}
static void fe_inv(fe* r, const fe* a, const field_t* F) {
    uint64_t e[4] = {F->p[0] - 2, F->p[1], F->p[2], F->p[3]};
    fe_pow(r, a, e, F);
}
static inline void fe_to_mont(fe* r, const fe* a, const field_t* F) { fe_mul(r, a, &F->r2, F); }
static inline void fe_from_mont(fe* r, const fe* a, const field_t* F) {
    fe one = {{1, 0, 0, 0}};
    fe_mul(r, a, &one, F);
}

/* ---------------------------------------------------------------- Fq2 = Fq[u]/(u^2+1) */
typedef struct { fe c0, c1; } fe2;
static inline void f2_add(fe2* r, const fe2* a, const fe2* b) { fe_add(&r->c0, &a->c0, &b->c0, &FQ); fe_add(&r->c1, &a->c1, &b->c1, &FQ); }
static inline void f2_sub(fe2* r, const fe2* a, const fe2* b) { fe_sub(&r->c0, &a->c0, &b->c0, &FQ); fe_sub(&r->c1, &a->c1, &b->c1, &FQ); }
static inline void f2_neg(fe2* r, const fe2* a) { fe_neg(&r->c0, &a->c0, &FQ); fe_neg(&r->c1, &a->c1, &FQ); }
static inline void f2_mul(fe2* r, const fe2* a, const fe2* b) {
    fe t0, t1, t2, s0, s1;
    fe_mul(&t0, &a->c0, &b->c0, &FQ); fe_mul(&t1, &a->c1, &b->c1, &FQ);
    fe_add(&s0, &a->c0, &a->c1, &FQ); fe_add(&s1, &b->c0, &b->c1, &FQ);
    fe_mul(&t2, &s0, &s1, &FQ);
    fe_sub(&r->c0, &t0, &t1, &FQ);
    fe_sub(&t2, &t2, &t0, &FQ); fe_sub(&r->c1, &t2, &t1, &FQ);
}
static inline void f2_sqr(fe2* r, const fe2* a) {
    fe s, d, t;
    fe_add(&s, &a->c0, &a->c1, &FQ); fe_sub(&d, &a->c0, &a->c1, &FQ);
    fe_mul(&t, &a->c0, &a->c1, &FQ);
    fe_mul(&r->c0, &s, &d, &FQ); fe_add(&r->c1, &t, &t, &FQ);
}
static void f2_inv(fe2* r, const fe2* a) {
    fe n, t;
    fe_sqr(&n, &a->c0, &FQ); fe_sqr(&t, &a->c1, &FQ); fe_add(&n, &n, &t, &FQ); fe_inv(&n, &n, &FQ);
    fe_mul(&r->c0, &a->c0, &n, &FQ); fe_mul(&t, &a->c1, &n, &FQ); fe_neg(&r->c1, &t, &FQ);
}
static inline int f2_is_zero(const fe2* a) { return fe_is_zero(&a->c0) && fe_is_zero(&a->c1); }
static inline int f2_eq(const fe2* a, const fe2* b) { return fe_eq(&a->c0, &b->c0) && fe_eq(&a->c1, &b->c1); }

/* ---------------------------------------------------------------- curves */
#define F_T fe
#define F_MUL(r, a, b) fe_mul(r, a, b, &FQ)
#define F_SQR(r, a) fe_sqr(r, a, &FQ)
#define F_ADD(r, a, b) fe_add(r, a, b, &FQ)
#define F_SUB(r, a, b) fe_sub(r, a, b, &FQ)
#define F_NEG(r, a) fe_neg(r, a, &FQ)
#define F_ISZERO(a) fe_is_zero(a)
#define F_EQ(a, b) fe_eq(a, b)
#define F_SET_ONE(r) (*(r) = FQ.one)
#define F_SET_ZERO(r) memset(r, 0, sizeof(fe))
#define F_INV(r, a) fe_inv(r, a, &FQ)
#define NAME(x) g1_##x
#include "curve_tmpl.h"
#undef F_T
#undef F_MUL
#undef F_SQR
#undef F_ADD
#undef F_SUB
#undef F_NEG
#undef F_ISZERO
#undef F_EQ
#undef F_SET_ONE
#undef F_SET_ZERO
#undef F_INV
#undef NAME

#define F_T fe2
#define F_MUL(r, a, b) f2_mul(r, a, b)
#define F_SQR(r, a) f2_sqr(r, a)
#define F_ADD(r, a, b) f2_add(r, a, b)
#define F_SUB(r, a, b) f2_sub(r, a, b)
#define F_NEG(r, a) f2_neg(r, a)
#define F_ISZERO(a) f2_is_zero(a)
#define F_EQ(a, b) f2_eq(a, b)
#define F_SET_ONE(r) do { (r)->c0 = FQ.one; memset(&(r)->c1, 0, sizeof(fe)); } while (0)
#define F_SET_ZERO(r) memset(r, 0, sizeof(fe2))
#define F_INV(r, a) f2_inv(r, a)
#define NAME(x) g2_##x
#include "curve_tmpl.h"

/* ---------------------------------------------------------------- NTT over Fr (Montgomery data) */
static fe fr_root(int bits) {          /* omega_bits = 5^((r-1)/2^bits) */
    fe five = {{5, 0, 0, 0}}, w;
    fe_to_mont(&five, &five, &FR);
    uint64_t e[4] = {FR.p[0] - 1, FR.p[1], FR.p[2], FR.p[3]};
    for (int s = 0; s < bits; s++) {   /* e >>= 1 */
        for (int i = 0; i < 4; i++) e[i] = (e[i] >> 1) | (i < 3 ? e[i + 1] << 63 : 0);
    }
    fe_pow(&w, &five, e, &FR);
    return w;
}

/* snarkjs polfield.js __fft: recursive radix-2, natural order in and out */
static void fft_rec(fe* out, const fe* in, size_t n, size_t stride, const fe* w, size_t wstride) {
    if (n == 1) { out[0] = in[0]; return; }
    size_t h = n / 2;
    fft_rec(out, in, h, stride * 2, w, wstride * 2);
    fft_rec(out + h, in + stride, h, stride * 2, w, wstride * 2);
    for (size_t i = 0; i < h; i++) {
        fe t;
        fe_mul(&t, &out[i + h], &w[i * wstride], &FR);
        fe a = out[i];
        fe_add(&out[i], &a, &t, &FR);
        fe_sub(&out[i + h], &a, &t, &FR);
    }
}

typedef struct { fe* a; const fe* w; size_t n; int bits, tid, nthreads; pthread_barrier_t* bar; } ntt_job;

/* iterative DIT on bit-reversed data; every level is split over the threads */
static void* ntt_worker(void* arg) {
    ntt_job* j = (ntt_job*)arg;
    size_t n = j->n, half = n / 2;
    for (int s = 0; s < j->bits; s++) {
        size_t h = (size_t)1 << s, step = half >> s;
        size_t lo = half * j->tid / j->nthreads, hi = half * (j->tid + 1) / j->nthreads;
        for (size_t b = lo; b < hi; b++) {
            size_t grp = b >> s, k = b & (h - 1);
            size_t i0 = (grp << (s + 1)) + k, i1 = i0 + h;
            fe t;
            fe_mul(&t, &j->a[i1], &j->w[k * step], &FR);
            fe u = j->a[i0];
            fe_add(&j->a[i0], &u, &t, &FR);
            fe_sub(&j->a[i1], &u, &t, &FR);
        }
        if (j->nthreads > 1) pthread_barrier_wait(j->bar);
    }
    return NULL;
}

/* in place; Montgomery data; inverse includes 1/n; mode 0 = recursive (snarkjs), 1 = iterative threaded */
static void ntt(fe* a, int bits, int inverse, int mode, int threads) {
    size_t n = (size_t)1 << bits;
    if (n == 1) return;
    fe w = fr_root(bits);
    if (inverse) fe_inv(&w, &w, &FR);
    fe* tw = (fe*)malloc(sizeof(fe) * (n / 2));
    tw[0] = FR.one;
    for (size_t i = 1; i < n / 2; i++) fe_mul(&tw[i], &tw[i - 1], &w, &FR);
    if (mode == 0) {
        fe* out = (fe*)malloc(sizeof(fe) * n);
        fft_rec(out, a, n, 1, tw, 1);
        memcpy(a, out, sizeof(fe) * n);
        free(out);
    } else {
        for (size_t i = 0; i < n; i++) {
            size_t r = 0;
            for (int b = 0; b < bits; b++) r |= ((i >> b) & 1) << (bits - 1 - b);
            if (r > i) { fe t = a[i]; a[i] = a[r]; a[r] = t; }
        }
        if (threads < 1) threads = 1;
        if (threads > 64) threads = 64;
        if (n < 4096) threads = 1;
        pthread_barrier_t bar;
        pthread_barrier_init(&bar, NULL, threads);
        pthread_t th[64]; ntt_job jobs[64];
        for (int t = 0; t < threads; t++) {
            jobs[t] = (ntt_job){a, tw, n, bits, t, threads, &bar};
            if (t) pthread_create(&th[t], NULL, ntt_worker, &jobs[t]);
        }
        ntt_worker(&jobs[0]);
        for (int t = 1; t < threads; t++) pthread_join(th[t], NULL);
        pthread_barrier_destroy(&bar);
    }
    if (inverse) {
        fe ninv = {{n, 0, 0, 0}};
        fe_to_mont(&ninv, &ninv, &FR); fe_inv(&ninv, &ninv, &FR);
        for (size_t i = 0; i < n; i++) fe_mul(&a[i], &a[i], &ninv, &FR);
    }
    free(tw);
}

/* ---------------------------------------------------------------- exported API (ctypes) */
static inline void rd_fe(fe* r, const uint8_t* p) { memcpy(r->v, p, 32); }

/* data: 2^bits x 32 B standard form; transformed in place (natural order).  coset: multiply by g^j
 * (forward) / g^-j (inverse), g = omega_{bits+1}. */
int oracle_ntt(uint8_t* data, int bits, int inverse, int coset, int mode, int threads) {
    size_t n = (size_t)1 << bits;
    fe* a = (fe*)malloc(sizeof(fe) * n);
    for (size_t i = 0; i < n; i++) { rd_fe(&a[i], data + 32 * i); fe_to_mont(&a[i], &a[i], &FR); }
    fe g = fr_root(bits + 1), s;
    if (coset && !inverse) {
        s = FR.one;
        for (size_t i = 0; i < n; i++) { fe_mul(&a[i], &a[i], &s, &FR); fe_mul(&s, &s, &g, &FR); }
    }
    ntt(a, bits, inverse, mode, threads);
    if (coset && inverse) {
        fe gi; fe_inv(&gi, &g, &FR);
        s = FR.one;
        for (size_t i = 0; i < n; i++) { fe_mul(&a[i], &a[i], &s, &FR); fe_mul(&s, &s, &gi, &FR); }
    }
    for (size_t i = 0; i < n; i++) { fe_from_mont(&a[i], &a[i], &FR); memcpy(data + 32 * i, a[i].v, 32); }
    free(a);
    return 0;
}

static void load_g1(g1_aff* out, const uint8_t* p, size_t n) {      /* Fq-M affine, x == 0 <=> infinity */
    for (size_t i = 0; i < n; i++) {
        rd_fe(&out[i].x, p + 64 * i); rd_fe(&out[i].y, p + 64 * i + 32);
        out[i].inf = fe_is_zero(&out[i].x);
    }
}
static void load_g2(g2_aff* out, const uint8_t* p, size_t n) {
    for (size_t i = 0; i < n; i++) {
        rd_fe(&out[i].x.c0, p + 128 * i); rd_fe(&out[i].x.c1, p + 128 * i + 32);
        rd_fe(&out[i].y.c0, p + 128 * i + 64); rd_fe(&out[i].y.c1, p + 128 * i + 96);
        out[i].inf = f2_is_zero(&out[i].x);
    }
}
static void store_g1_std(uint8_t* out, const g1_jac* p) {
    g1_aff a; g1_to_affine(&a, p);
    if (a.inf) { memset(out, 0, 64); return; }
    fe t; fe_from_mont(&t, &a.x, &FQ); memcpy(out, t.v, 32); fe_from_mont(&t, &a.y, &FQ); memcpy(out + 32, t.v, 32);
}
static void store_g2_std(uint8_t* out, const g2_jac* p) {
    g2_aff a; g2_to_affine(&a, p);
    if (a.inf) { memset(out, 0, 128); return; }
    fe t;
    fe_from_mont(&t, &a.x.c0, &FQ); memcpy(out, t.v, 32); fe_from_mont(&t, &a.x.c1, &FQ); memcpy(out + 32, t.v, 32);
    fe_from_mont(&t, &a.y.c0, &FQ); memcpy(out + 64, t.v, 32); fe_from_mont(&t, &a.y.c1, &FQ); memcpy(out + 96, t.v, 32);
}

/* points: affine Fq-M (64 B G1 / 128 B G2); scalars: 32 B standard form; out: affine standard form */
int oracle_msm(int group, const uint8_t* points, const uint8_t* scalars, size_t n, uint8_t* out, int mode, int threads) {
    const uint64_t (*sc)[4] = (const uint64_t (*)[4])scalars;
    if (group == 1) {
        g1_aff* pts = (g1_aff*)malloc(sizeof(g1_aff) * (n ? n : 1));
        load_g1(pts, points, n);
        g1_jac r; g1_msm(&r, pts, sc, n, mode, threads);
        store_g1_std(out, &r); free(pts);
    } else {
        g2_aff* pts = (g2_aff*)malloc(sizeof(g2_aff) * (n ? n : 1));
        load_g2(pts, points, n);
        g2_jac r; g2_msm(&r, pts, sc, n, mode, threads);
        store_g2_std(out, &r); free(pts);
    }
    return 0;
}

static inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }

/* A_T / B_T from one pols section (binarify.ts:104-113); out Montgomery */
static size_t eval_pols(fe* out, size_t m, const uint8_t* pk, size_t off, uint32_t n, const fe* w_mont) {
    memset(out, 0, sizeof(fe) * m);
    for (uint32_t s = 0; s < n; s++) {
        uint32_t k = rd32(pk + off); off += 4;
        for (uint32_t j = 0; j < k; j++) {
            uint32_t row = rd32(pk + off);
            fe c, t; rd_fe(&c, pk + off + 4);
            fe_mul(&t, &c, &w_mont[s], &FR);
            fe_add(&out[row], &out[row], &t, &FR);
            off += 36;
        }
    }
    return off;
}

/* websnark calcH: A, B on the 2m domain (even slots given, odd slots via iNTT_m + shifted NTT_m), pointwise multiply,
 * iNTT_2m, upper half (SURVEY.md B.4 ii).  at, bt: the m = 2^bits evaluations A_T, B_T, Montgomery (not modified);
 * h_out: m x 32 B standard form. */
static void calc_h(const fe* at, const fe* bt, int bits, uint8_t* h_out, int mode, int threads) {
    const size_t m = (size_t)1 << bits;
    fe* ao = (fe*)malloc(sizeof(fe) * m); fe* bo = (fe*)malloc(sizeof(fe) * m);
    fe* ab = (fe*)malloc(sizeof(fe) * 2 * m);
    memcpy(ao, at, sizeof(fe) * m); memcpy(bo, bt, sizeof(fe) * m);
    ntt(ao, bits, 1, mode, threads); ntt(bo, bits, 1, mode, threads);
    fe g = fr_root(bits + 1), s = FR.one;
    for (size_t i = 0; i < m; i++) { fe_mul(&ao[i], &ao[i], &s, &FR); fe_mul(&bo[i], &bo[i], &s, &FR); fe_mul(&s, &s, &g, &FR); }
    ntt(ao, bits, 0, mode, threads); ntt(bo, bits, 0, mode, threads);
    for (size_t i = 0; i < m; i++) { fe_mul(&ab[2 * i], &at[i], &bt[i], &FR); fe_mul(&ab[2 * i + 1], &ao[i], &bo[i], &FR); }
    ntt(ab, bits + 1, 1, mode, threads);
    for (size_t i = 0; i < m; i++) { fe t; fe_from_mont(&t, &ab[m + i], &FR); memcpy(h_out + 32 * i, t.v, 32); }
    free(ao); free(bo); free(ab);
}

/* h of calcH from the evaluations alone (the GPU's zkr_h_from_evals_dev, computed by websnark's method rather than its
 * L/U split).  at32, bt32: 2^bits x 32 B standard form; h_out: 2^bits x 32 B standard form.  mode, threads: as ntt. */
int oracle_h_from_evals(const uint8_t* at32, const uint8_t* bt32, int bits, uint8_t* h_out, int mode, int threads) {
    const size_t m = (size_t)1 << bits;
    fe* at = (fe*)malloc(sizeof(fe) * m); fe* bt = (fe*)malloc(sizeof(fe) * m);
    for (size_t i = 0; i < m; i++) {
        rd_fe(&at[i], at32 + 32 * i); fe_to_mont(&at[i], &at[i], &FR);
        rd_fe(&bt[i], bt32 + 32 * i); fe_to_mont(&bt[i], &bt[i], &FR);
    }
    calc_h(at, bt, bits, h_out, mode, threads);
    free(at); free(bt);
    return 0;
}

/* websnark groth16GenProof restated.  pk: binarifyProvingKey bytes; witness: n x 32 B standard form;
 * r32, s32: blinding scalars (standard form) or NULL for 0; out: 256 B proof (include/zkr.h layout).
 * mode 0: snarkjs-structured arithmetic (per-point double-and-add, recursive FFT), single thread;
 * mode 1: Pippenger + iterative NTT on `threads` threads.  h_out (optional): m x 32 B std-form h. */
int oracle_prove(const uint8_t* pk, size_t pk_len, const uint8_t* witness, size_t n_signals, const uint8_t* r32,
                 const uint8_t* s32, uint8_t* out, int mode, int threads, uint8_t* h_out) {
    if (pk_len < 488) return -2;
    uint32_t n = rd32(pk), l = rd32(pk + 4), m = rd32(pk + 8);
    uint32_t pA = rd32(pk + 12), pB = rd32(pk + 16), pPA = rd32(pk + 20), pPB1 = rd32(pk + 24), pPB2 = rd32(pk + 28),
             pPC = rd32(pk + 32), pPH = rd32(pk + 36);
    if (n_signals != n) return -1;
    int bits = 0; while (((uint32_t)1 << bits) < m) bits++;
    (void)pPA;
    /* witness -> Montgomery (websnark fft_toMontgomeryN) */
    fe* wm = (fe*)malloc(sizeof(fe) * n);
    for (uint32_t i = 0; i < n; i++) { rd_fe(&wm[i], witness + 32 * (size_t)i); fe_to_mont(&wm[i], &wm[i], &FR); }
    /* calcH */
    fe* at = (fe*)malloc(sizeof(fe) * m); fe* bt = (fe*)malloc(sizeof(fe) * m);
    eval_pols(at, m, pk, pA, n, wm);
    eval_pols(bt, m, pk, pB, n, wm);
    uint64_t (*h)[4] = (uint64_t (*)[4])malloc(32 * (size_t)m);
    calc_h(at, bt, bits, (uint8_t*)h, mode, threads);
    if (h_out) memcpy(h_out, h, 32 * (size_t)m);
    free(at); free(bt); free(wm);
    /* multiexps */
    const uint64_t (*w)[4] = (const uint64_t (*)[4])witness;
    g1_aff* p1 = (g1_aff*)malloc(sizeof(g1_aff) * (n > m ? n : m));
    g1_jac sa, sb1, sc, sh; g2_jac sb2;
    load_g1(p1, pk + pPA, n); g1_msm(&sa, p1, w, n, mode, threads);
    load_g1(p1, pk + pPB1, n); g1_msm(&sb1, p1, w, n, mode, threads);
    load_g1(p1, pk + pPC, n - l - 1); g1_msm(&sc, p1, w + l + 1, n - l - 1, mode, threads);
    load_g1(p1, pk + pPH, m); g1_msm(&sh, p1, (const uint64_t (*)[4])h, m, mode, threads);
    g2_aff* p2 = (g2_aff*)malloc(sizeof(g2_aff) * n);
    load_g2(p2, pk + pPB2, n); g2_msm(&sb2, p2, w, n, mode, threads);
    free(p1); free(p2); free(h);
    /* blinding + assembly (SURVEY.md B.2) */
    uint64_t rr[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0}, rs[4];
    if (r32) memcpy(rr, r32, 32);
    if (s32) memcpy(ss, s32, 32);
    { fe a, b, c; memcpy(a.v, rr, 32); memcpy(b.v, ss, 32); fe_to_mont(&a, &a, &FR); fe_to_mont(&b, &b, &FR);
      fe_mul(&c, &a, &b, &FR); fe_from_mont(&c, &c, &FR); memcpy(rs, c.v, 32); }
    g1_aff alfa1, beta1, delta1; g2_aff beta2, delta2;
    load_g1(&alfa1, pk + 40, 1); load_g1(&beta1, pk + 104, 1); load_g1(&delta1, pk + 168, 1);
    load_g2(&beta2, pk + 232, 1); load_g2(&delta2, pk + 360, 1);
    g1_jac d1j, t, pia, pib1, pic; g2_jac d2j, t2, pib;
    g1_jset_inf(&d1j); g1_jmadd(&d1j, &d1j, &delta1);
    g2_jset_inf(&d2j); g2_jmadd(&d2j, &d2j, &delta2);
    g1_jmadd(&pia, &sa, &alfa1); g1_jmul(&t, &d1j, rr); g1_jadd(&pia, &pia, &t);
    g2_jmadd(&pib, &sb2, &beta2); g2_jmul(&t2, &d2j, ss); g2_jadd(&pib, &pib, &t2);
    g1_jmadd(&pib1, &sb1, &beta1); g1_jmul(&t, &d1j, ss); g1_jadd(&pib1, &pib1, &t);
    g1_jadd(&pic, &sc, &sh);
    g1_jmul(&t, &pia, ss); g1_jadd(&pic, &pic, &t);
    g1_jmul(&t, &pib1, rr); g1_jadd(&pic, &pic, &t);
    g1_jmul(&t, &d1j, rs); g1_jneg(&t, &t); g1_jadd(&pic, &pic, &t);
    store_g1_std(out, &pia); store_g2_std(out + 64, &pib); store_g1_std(out + 192, &pic);
    return 0;
}

/* out[i] = base + i * step, affine Fq-M bytes (64 B G1 / 128 B G2; infinity = zeros); base, step affine Fq-M.
 * With base = a0 G and step = d G this is P_i = (a0 + i d) G of SURVEY.md 8(d) config 3, made on the host. */
int oracle_ap_points(int group, const uint8_t* base, const uint8_t* step, size_t n, uint8_t* out) {
    if (group == 1) {
        g1_aff b, s, *o = (g1_aff*)malloc(sizeof(g1_aff) * (n ? n : 1));
        load_g1(&b, base, 1); load_g1(&s, step, 1);
        g1_ap_points(o, &b, &s, n);
        for (size_t i = 0; i < n; i++) {
            if (o[i].inf) { memset(out + 64 * i, 0, 64); continue; }
            memcpy(out + 64 * i, o[i].x.v, 32); memcpy(out + 64 * i + 32, o[i].y.v, 32);
        }
        free(o);
    } else {
        g2_aff b, s, *o = (g2_aff*)malloc(sizeof(g2_aff) * (n ? n : 1));
        load_g2(&b, base, 1); load_g2(&s, step, 1);
        g2_ap_points(o, &b, &s, n);
        for (size_t i = 0; i < n; i++) {
            if (o[i].inf) { memset(out + 128 * i, 0, 128); continue; }
            memcpy(out + 128 * i, o[i].x.c0.v, 32); memcpy(out + 128 * i + 32, o[i].x.c1.v, 32);
            memcpy(out + 128 * i + 64, o[i].y.c0.v, 32); memcpy(out + 128 * i + 96, o[i].y.c1.v, 32);
        }
        free(o);
    }
    return 0;
}

/* Toxic-waste exponent sums (oracle/groth16.py exponent_check_flat, restated): for one sparse matrix given as
 * (sig, row, cid) triplets with coefficients pool[cid],
 *     tot  = sum_e w[sig_e] pool[cid_e] L_{row_e}(tau),     priv = the same over entries with sig_e > n_public,
 * L_c(tau) = omega^c (tau^m - 1) / (m (tau - omega^c)) on the domain <omega_m> (lagrange_at).  No MSM / NTT code.
 * w: n x 32 B, pool: n_pool x 32 B, tau32, out: standard form.  One shared inversion (Montgomery's trick). */
int oracle_exponent_sums(int log_m, const uint8_t* tau32, const uint8_t* w, const uint8_t* pool, size_t n_pool,
                         const uint32_t* sig, const uint32_t* row, const uint32_t* cid, size_t nnz, uint32_t n_public,
                         uint8_t* tot32, uint8_t* priv32) {
    const size_t m = (size_t)1 << log_m;
    fe tau, om = fr_root(log_m), zt, k, minv, t;
    rd_fe(&tau, tau32); fe_to_mont(&tau, &tau, &FR);
    zt = tau;
    for (int i = 0; i < log_m; i++) fe_sqr(&zt, &zt, &FR);
    fe_sub(&zt, &zt, &FR.one, &FR);
    fe mm = {{(uint64_t)m, 0, 0, 0}};
    fe_to_mont(&mm, &mm, &FR); fe_inv(&minv, &mm, &FR);
    fe_mul(&k, &zt, &minv, &FR);
    fe* lag = (fe*)malloc(sizeof(fe) * m);        /* tau - omega^c, then L_c(tau), Montgomery */
    fe* pre = (fe*)malloc(sizeof(fe) * m);
    fe* wc = (fe*)malloc(sizeof(fe) * m);
    fe cur = FR.one, acc = FR.one;
    for (size_t c = 0; c < m; c++) {
        wc[c] = cur;
        fe_sub(&lag[c], &tau, &cur, &FR);
        pre[c] = acc;
        fe_mul(&acc, &acc, &lag[c], &FR);
        fe_mul(&cur, &cur, &om, &FR);
    }
    fe inv; fe_inv(&inv, &acc, &FR);
    for (size_t c = m; c-- > 0;) {
        fe di; fe_mul(&di, &inv, &pre[c], &FR);
        fe_mul(&inv, &inv, &lag[c], &FR);
        fe_mul(&t, &k, &wc[c], &FR);
        fe_mul(&lag[c], &t, &di, &FR);
    }
    fe* pm = (fe*)malloc(sizeof(fe) * (n_pool ? n_pool : 1));
    for (size_t i = 0; i < n_pool; i++) { rd_fe(&pm[i], pool + 32 * i); fe_to_mont(&pm[i], &pm[i], &FR); }
    fe tot = {{0, 0, 0, 0}}, priv = {{0, 0, 0, 0}};
    for (size_t e = 0; e < nnz; e++) {
        fe ws; rd_fe(&ws, w + 32 * (size_t)sig[e]);
        fe_mul(&t, &ws, &pm[cid[e]], &FR);        /* standard x Montgomery -> standard */
        fe_mul(&t, &t, &lag[row[e]], &FR);
        fe_add(&tot, &tot, &t, &FR);
        if (sig[e] > n_public) fe_add(&priv, &priv, &t, &FR);
    }
    memcpy(tot32, tot.v, 32); memcpy(priv32, priv.v, 32);
    free(pm); free(wc); free(pre); free(lag);
    return 0;
}

/* Horner evaluation over Fr: out = sum_j coeffs[j] x^j; coeffs n x 32 B, x, out 32 B, all standard form.
 * The NTT check of SURVEY.md 8(d) config 4 ("Horner evaluation at 8 random points vs. transformed values"). */
int oracle_horner(const uint8_t* coeffs, size_t n, const uint8_t* x32, uint8_t* out32) {
    fe x, acc = {{0, 0, 0, 0}}, c;
    rd_fe(&x, x32); fe_to_mont(&x, &x, &FR);
    for (size_t j = n; j-- > 0;) {
        fe_mul(&acc, &acc, &x, &FR);          /* standard-form acc times Montgomery x stays standard form */
        rd_fe(&c, coeffs + 32 * j);
        fe_add(&acc, &acc, &c, &FR);
    }
    memcpy(out32, acc.v, 32);
    return 0;
}

/* affine point addition / scalar multiplication (k: 32 B standard form), points Fq-M affine bytes, infinity = zeros:
 * the operations of the alt_bn128 ecAdd / ecMul precompiles TxVerifier.sol:59-88 calls (EIP-196 known answers) */
int oracle_g1_add(const uint8_t* p, const uint8_t* q, uint8_t* out) {
    g1_aff a, b; load_g1(&a, p, 1); load_g1(&b, q, 1);
    g1_jac j; j.x = a.x; j.y = a.y; j.z = FQ.one; if (a.inf) g1_jset_inf(&j);
    g1_jmadd(&j, &j, &b);
    g1_aff r; g1_to_affine(&r, &j);
    if (r.inf) { memset(out, 0, 64); return 0; }
    memcpy(out, r.x.v, 32); memcpy(out + 32, r.y.v, 32);
    return 0;
}
int oracle_g1_mul(const uint8_t* p, const uint8_t* k32, uint8_t* out) {
    g1_aff a; load_g1(&a, p, 1);
    uint64_t k[4]; memcpy(k, k32, 32);
    g1_jac j, r; j.x = a.x; j.y = a.y; j.z = FQ.one; if (a.inf) g1_jset_inf(&j);
    g1_jmul(&r, &j, k);
    g1_aff o; g1_to_affine(&o, &r);
    if (o.inf) { memset(out, 0, 64); return 0; }
    memcpy(out, o.x.v, 32); memcpy(out + 32, o.y.v, 32);
    return 0;
}

/* element-wise Montgomery product in Fq (field = 0) or Fr (field = 1): KAT hook for the tests */
int oracle_field_mul(int field, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n) {
    const field_t* F = field ? &FR : &FQ;
    for (size_t i = 0; i < n; i++) {
        fe x, y, z; rd_fe(&x, a + 32 * i); rd_fe(&y, b + 32 * i);
        fe_mul(&z, &x, &y, F); memcpy(out + 32 * i, z.v, 32);
    }
    return 0;
}
