// Short-Weierstrass (a = 0) point arithmetic in XYZZ coordinates, templated on the coordinate
// field (Fq for G1, Fq2 for G2).  Replaces snarkjs GCurve / websnark g1m_*, g2m_* used by the
// five multiexps of groth16GenProof (/root/reference/operator/src/snarks/common.ts:29).
//
//   XYZZ:  x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2;   identity <=> ZZ == 0  (all-zero words, so
//   cudaMemset(0) produces an array of identities).
//   mixed add 8M+2S, full add 12M+2S, doubling 6M+3S  (EFD madd-2008-s / add-2008-s / dbl-2008-s-1).
// Exceptional inputs (P == Q, P == -Q, identity operands) are handled, not assumed away.
#pragma once
#include "fp.cuh"

#if !defined(__CUDACC__) && !defined(__noinline__)
#define __noinline__
#endif
#ifndef ZKR_LAZY_TAIL
// 1 (default): the full XYZZ addition and the doublings (bucket gather / reduction, blinding, tails) use the lazily reduced
// forms as well; 0 keeps the round-1 arithmetic there (A/B: profiles/r02_lazy_reduction_ab.json, build.py ZKR_BUILD_VARIANT)
#define ZKR_LAZY_TAIL 1
#endif

namespace zkr {

template <class F>
struct Affine {
    F x, y;
    // websnark loader rule (binarify.ts:92-95 drops z): x == 0 <=> point at infinity
    __device__ __forceinline__ bool is_inf() const { return x.is_zero(); }
    static __device__ __forceinline__ Affine load(const void* p) {
        return {F::load(p), F::load(reinterpret_cast<const char*>(p) + sizeof(F))};
    }
    static __device__ __forceinline__ Affine load_ro(const void* p) {
        return {F::load_ro(p), F::load_ro(reinterpret_cast<const char*>(p) + sizeof(F))};
    }
    __device__ __forceinline__ void store(void* p) const {
        x.store(p);
        y.store(reinterpret_cast<char*>(p) + sizeof(F));
    }
    __device__ __forceinline__ Affine neg() const { return {x, y.neg()}; }
};

template <class F>
struct XYZZ {
    F x, y, zz, zzz;

    static __device__ __forceinline__ XYZZ identity() { return {F::zero(), F::zero(), F::zero(), F::zero()}; }
    static __device__ __forceinline__ XYZZ from_affine(const Affine<F>& p) {
        if (p.is_inf()) return identity();
        return {p.x, p.y, F::one(), F::one()};
    }
    __device__ __forceinline__ bool is_inf() const { return zz.is_zero(); }
    __device__ __forceinline__ XYZZ neg() const { return {x, y.neg(), zz, zzz}; }

    static __device__ __forceinline__ XYZZ load(const void* p) {
        const char* c = reinterpret_cast<const char*>(p);
        return {F::load(c), F::load(c + sizeof(F)), F::load(c + 2 * sizeof(F)), F::load(c + 3 * sizeof(F))};
    }
    __device__ __forceinline__ void store(void* p) const {
        char* c = reinterpret_cast<char*>(p);
        x.store(c);
        y.store(c + sizeof(F));
        zz.store(c + 2 * sizeof(F));
        zzz.store(c + 3 * sizeof(F));
    }

    // 2 * (affine point)
    static __device__ __forceinline__ XYZZ dbl_affine(const Affine<F>& p) {
        if (p.y.is_zero()) return identity();
        F u = p.y.dbl();
        F v = u.sqr();
        F w = u * v;
        F s = p.x * v;
        F xx = p.x.sqr();
        F m = xx.dbl() + xx;
        F x3 = m.sqr() - s.dbl();
#if ZKR_LAZY_TAIL
        F y3 = F::msub(m, s - x3, w, p.y);
#else
        F y3 = m * (s - x3) - w * p.y;
#endif
        return {x3, y3, v, w};
    }

    __device__ __forceinline__ XYZZ dbl() const {
        if (is_inf() || y.is_zero()) return identity();
        F u = y.dbl();
        F v = u.sqr();
        F w = u * v;
        F s = x * v;
        F xx = x.sqr();
        F m = xx.dbl() + xx;
        F x3 = m.sqr() - s.dbl();
#if ZKR_LAZY_TAIL
        F y3 = F::msub(m, s - x3, w, y);
        return {x3, y3, F::mul_l(v, zz), F::mul_l(w, zzz)};
#else
        F y3 = m * (s - x3) - w * y;
        return {x3, y3, v * zz, w * zzz};
#endif
    }

    // this += affine q  (q must not be infinity)
    __device__ __forceinline__ void madd(const Affine<F>& q) {
        if (is_inf()) {
            x = q.x; y = q.y; zz = F::one(); zzz = F::one();
            return;
        }
        F p = q.x * zz - x;
        F r = q.y * zzz - y;
        if (p.is_zero()) {
            if (r.is_zero()) *this = dbl_affine(q);
            else *this = identity();
            return;
        }
        F pp = p.sqr();
        F ppp = p * pp;
        F qq = x * pp;
        F x3 = r.sqr() - ppp - qq.dbl();
        y = r * (qq - x3) - y * ppp;
        x = x3;
        zz = zz * pp;
        zzz = zzz * ppp;
    }

    // Same addition with the sums of products reduced once (fp.cuh "sums of products"): y3 = r (q - x3) - y ppp is one
    // two-product pass for G1 (200 instead of 272 multiplier instructions, one subtraction and one final correction
    // fewer) and two four-product passes for G2; G2's six plain products use the schoolbook-lazy Fq2::mul_l.
    // Results are canonical and bit-identical to madd().
    // FSQ: the two squarings (p^2, r^2) through Fp::sqr_fast (100 instead of 128 wide multiplies each; G1 only)
    template <bool FSQ = false>
    __device__ __forceinline__ void madd_lazy(const Affine<F>& q) {
        if (is_inf()) {
            x = q.x; y = q.y; zz = F::one(); zzz = F::one();
            return;
        }
        F p = F::mul_l(q.x, zz) - x;
        F r = F::mul_l(q.y, zzz) - y;
        if (p.is_zero()) {
            if (r.is_zero()) *this = dbl_affine(q);
            else *this = identity();
            return;
        }
        F pp = FSQ ? p.sqr_fast() : p.sqr();
        F ppp = F::mul_l(p, pp);
        F qq = F::mul_l(x, pp);
        F x3 = (FSQ ? r.sqr_fast() : r.sqr()) - ppp - qq.dbl();
        y = F::msub(r, qq - x3, y, ppp);
        x = x3;
        zz = F::mul_l(zz, pp);
        zzz = F::mul_l(zzz, ppp);
    }

    // this += o
    __device__ __forceinline__ void add(const XYZZ& o) {
        if (o.is_inf()) return;
        if (is_inf()) { *this = o; return; }
#if ZKR_LAZY_TAIL
        F u1 = F::mul_l(x, o.zz), u2 = F::mul_l(o.x, zz);
        F s1 = F::mul_l(y, o.zzz), s2 = F::mul_l(o.y, zzz);
#else
        F u1 = x * o.zz, u2 = o.x * zz;
        F s1 = y * o.zzz, s2 = o.y * zzz;
#endif
        F p = u2 - u1;
        F r = s2 - s1;
        if (p.is_zero()) {
            if (r.is_zero()) *this = dbl();
            else *this = identity();
            return;
        }
        F pp = p.sqr();
#if ZKR_LAZY_TAIL          // sums of products reduced once, Fq2 products schoolbook-lazy (see madd_lazy); same words out
        F ppp = F::mul_l(p, pp);
        F qq = F::mul_l(u1, pp);
        F x3 = r.sqr() - ppp - qq.dbl();
        y = F::msub(r, qq - x3, s1, ppp);
        x = x3;
        zz = F::mul_l(F::mul_l(zz, o.zz), pp);
        zzz = F::mul_l(F::mul_l(zzz, o.zzz), ppp);
#else
        F ppp = p * pp;
        F qq = u1 * pp;
        F x3 = r.sqr() - ppp - qq.dbl();
        y = r * (qq - x3) - s1 * ppp;
        x = x3;
        zz = zz * o.zz * pp;
        zzz = zzz * o.zzz * ppp;
#endif
    }

    // affine, Montgomery form; identity -> (0, 0)
    __device__ __forceinline__ Affine<F> to_affine() const {
        if (is_inf()) return {F::zero(), F::zero()};
        // 1/zzz gives both: 1/zz = (1/zzz)^2 * zz^2 ... cheaper: one inversion of zzz, then
        // 1/zz = zzz^-2 * zz^2  (since zz^3 = zzz^2  =>  zz^-1 = zz^2 * zzz^-2)
        F iz3 = zzz.inverse();
        F iz2 = iz3.sqr() * zz.sqr();
        return {x * iz2, y * iz3};
    }
    // same, with the variable-time inversion of fp_inv.cuh: single-thread tails only (k_finish)
    __device__ __forceinline__ Affine<F> to_affine_vartime() const {
        if (is_inf()) return {F::zero(), F::zero()};
        F iz3 = zzz.inverse_vartime();
        F iz2 = iz3.sqr() * zz.sqr();
        return {x * iz2, y * iz3};
    }
};

using G1Affine = Affine<Fq>;
using G2Affine = Affine<Fq2>;
using G1XYZZ = XYZZ<Fq>;
using G2XYZZ = XYZZ<Fq2>;

// Out-of-line helpers for cold paths (block-level bucket reduction).  They are strictly
// MEMORY-TO-MEMORY: every pointer must address shared or global memory and all big values live
// inside the callee.  Passing 256-byte structs across a device call boundary (by value, or as
// pointers to the caller's locals) produced wrong results with nvcc/ptxas 12.9 on sm_100a -- see
// DESIGN.md "toolchain notes" and tools/scratch/variants.cu for the reproducer.
template <class F>
__device__ __noinline__ void xyzz_add_mem(XYZZ<F>* dst, const XYZZ<F>* a, const XYZZ<F>* b) {
    XYZZ<F> x = *a;
    x.add(*b);
    *dst = x;
}
template <class F>
__device__ __noinline__ void xyzz_dbl_mem(XYZZ<F>* dst) {
    XYZZ<F> x = *dst;
    *dst = x.dbl();
}

template <class F>
__device__ __forceinline__ Affine<F> generator();
template <>
__device__ __forceinline__ Affine<Fq> generator<Fq>() {   // (1, 2): TxVerifier.sol:24-26
    Fq one = Fq::one();
    return {one, one + one};
}
template <>
__device__ __forceinline__ Affine<Fq2> generator<Fq2>() {   // TxVerifier.sol:30-35 (real part second there)
    const uint32_t x0[8] = {0xd992f6edu, 0x46debd5cu, 0xf75edaddu, 0x674322d4u, 0x5e5c4479u, 0x426a0066u, 0x121f1e76u, 0x1800deefu};
    const uint32_t x1[8] = {0xaef312c2u, 0x97e485b7u, 0x35a9e712u, 0xf1aa4933u, 0x31fb5d25u, 0x7260bfb7u, 0x920d483au, 0x198e9393u};
    const uint32_t y0[8] = {0x66fa7daau, 0x4ce6cc01u, 0x0c43d37bu, 0xe3d1e769u, 0x8dcb408fu, 0x4aab7180u, 0xdb8c6debu, 0x12c85ea5u};
    const uint32_t y1[8] = {0xd122975bu, 0x55acdadcu, 0x70b38ef3u, 0xbc4b3133u, 0x690c3395u, 0xec9e99adu, 0x585ff075u, 0x090689d0u};
    Fq a, b, c, d;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        a.v[i] = x0[i];
        b.v[i] = x1[i];
        c.v[i] = y0[i];
        d.v[i] = y1[i];
    }
    return {{a.to_mont(), b.to_mont()}, {c.to_mont(), d.to_mont()}};
}

// k * p, k a 256-bit standard-form integer (LSB-first double-and-add); O(1) uses per proof only.
template <class F>
__device__ __forceinline__ XYZZ<F> scalar_mul(XYZZ<F> p, Fr k) {
    XYZZ<F> acc = XYZZ<F>::identity(), base = p;
    int top = 255;
    while (top >= 0 && !((k.v[top >> 5] >> (top & 31)) & 1)) top--;
    for (int i = 0; i <= top; i++) {
        if ((k.v[i >> 5] >> (i & 31)) & 1) acc.add(base);
        if (i < top) base = base.dbl();
    }
    return acc;
}

}  // namespace zkr
