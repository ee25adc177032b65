// Groth16 verification for the proof generator's self-check (SURVEY.md 8(f) rank 2).
//
// Replaces snarkjs `groth.isValid(verifyingKey, proof, publicSignals)` at
// /root/reference/operator/src/snarks/common.ts:30-34, which the reference runs after EVERY proof on the JS
// BigInt path (seconds) and which would dominate createProofGenerator once the prove itself takes milliseconds.
// The predicate is the on-chain one, /root/reference/contracts/contracts/TxVerifier.sol:258-276:
//     vk_x = IC[0] + sum_i input[i] * IC[i+1]                       (inputs < r, :265)
//     e(-A, B) * e(alfa1, beta2) * e(vk_x, gamma2) * e(C, delta2) == 1   (pairingProd4, :269-274)
// Split of work:
//   * vk_x is an l-term G1 MSM over bases fixed per circuit (l = 73 for tx.circom, 577 / 2305 at the scaled
//     sizes): it runs on the GPU through the same window-precomputed bucket MSM as the prover (zkr_bases_load
//     once per verifying key, zkr_msm per proof) -- on the host it would cost l double-and-add multiplications.
//   * the pairing product is O(1) work with no data parallelism (4 Miller loops sharing one accumulator, one
//     final exponentiation): it runs on the host core that issued the call, 4 x 64-bit Montgomery limbs,
//     ~2 ms, while the GPU is free for the next proof.  Same split as the reference (pairings on the CPU).
// Fq12 = Fq2[w]/(w^6 - xi), xi = 9 + u; optimal-ate Miller loop over 6x+2 with the twist points in homogeneous
// projective coordinates (no inversion in the loop; the first, affine version with per-step batched inversions is
// kept behind ZKR_PAIRING_AFFINE=1 as a cross-check), two Frobenius line additions, final exponentiation with the
// BN hard part of Scott et al. (exponentiations by x with cyclotomic squarings, Frobenius maps).
#include <immintrin.h>

#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "host_ec.cuh"
#include "keyjson_iface.cuh"

namespace zkr {
namespace pr {

typedef unsigned __int128 u128;

// ------------------------------------------------------------------------------------------------ Fq
struct Fq {
    uint64_t v[4];
};
const uint64_t kP[4] = {0x3c208c16d87cfd47ull, 0x97816a916871ca8dull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
const uint64_t kInv = 0x87d20782e4866389ull;
const Fq kOne = {{0xd35d438dc58f0d9dull, 0x0a78eb28f5c70b3dull, 0x666ea36f7879462cull, 0x0e0a77c19a07df2full}};
const Fq kR2 = {{0xf32cfc5b538afa89ull, 0xb5e71911d44501fbull, 0x47ab1eff0a417ff6ull, 0x06d89f71cab8351full}};
const Fq kZero = {{0, 0, 0, 0}};
// scalar field modulus r (TxVerifier.sol:259), for the G2 subgroup check
const uint64_t kRmod[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};

inline bool is_zero(const Fq& a) { return (a.v[0] | a.v[1] | a.v[2] | a.v[3]) == 0; }
inline bool eq(const Fq& a, const Fq& b) {
    return ((a.v[0] ^ b.v[0]) | (a.v[1] ^ b.v[1]) | (a.v[2] ^ b.v[2]) | (a.v[3] ^ b.v[3])) == 0;
}
inline bool geq_p(const uint64_t* a) {
    for (int i = 3; i >= 0; i--)
        if (a[i] != kP[i]) return a[i] > kP[i];
    return true;
}
// r = t - p if t >= p else t   (t < 2p), branch-free adc / sbb chains
inline Fq cond_sub_p(uint64_t t0, uint64_t t1, uint64_t t2, uint64_t t3) {
    unsigned long long s0, s1, s2, s3;
    unsigned char bw = _subborrow_u64(0, t0, kP[0], &s0);
    bw = _subborrow_u64(bw, t1, kP[1], &s1);
    bw = _subborrow_u64(bw, t2, kP[2], &s2);
    bw = _subborrow_u64(bw, t3, kP[3], &s3);
    const uint64_t keep = 0 - (uint64_t)bw;      // all ones if t < p
    return {{(t0 & keep) | (s0 & ~keep), (t1 & keep) | (s1 & ~keep), (t2 & keep) | (s2 & ~keep), (t3 & keep) | (s3 & ~keep)}};
}
inline Fq add(const Fq& a, const Fq& b) {      // a + b < 2p < 2^255: no carry out of the top word
    unsigned long long t0, t1, t2, t3;
    unsigned char c = _addcarry_u64(0, a.v[0], b.v[0], &t0);
    c = _addcarry_u64(c, a.v[1], b.v[1], &t1);
    c = _addcarry_u64(c, a.v[2], b.v[2], &t2);
    _addcarry_u64(c, a.v[3], b.v[3], &t3);
    return cond_sub_p(t0, t1, t2, t3);
}
inline Fq sub(const Fq& a, const Fq& b) {
    unsigned long long t0, t1, t2, t3;
    unsigned char bw = _subborrow_u64(0, a.v[0], b.v[0], &t0);
    bw = _subborrow_u64(bw, a.v[1], b.v[1], &t1);
    bw = _subborrow_u64(bw, a.v[2], b.v[2], &t2);
    bw = _subborrow_u64(bw, a.v[3], b.v[3], &t3);
    const uint64_t m = 0 - (uint64_t)bw;          // all ones if a < b: add p back
    unsigned long long r0, r1, r2, r3;
    unsigned char c = _addcarry_u64(0, t0, kP[0] & m, &r0);
    c = _addcarry_u64(c, t1, kP[1] & m, &r1);
    c = _addcarry_u64(c, t2, kP[2] & m, &r2);
    _addcarry_u64(c, t3, kP[3] & m, &r3);
    return {{r0, r1, r2, r3}};
}
inline Fq neg(const Fq& a) { return is_zero(a) ? a : sub(kZero, a); }
inline Fq dbl(const Fq& a) { return add(a, a); }
// CIOS with the reduction row fused into the product row; q < 2^254 leaves the top word headroom, so the
// running value fits 4 words + the two carries added at the end of each row
inline Fq mul(const Fq& a, const Fq& b) {
    uint64_t t0 = 0, t1 = 0, t2 = 0, t3 = 0;
#pragma GCC unroll 4
    for (int i = 0; i < 4; i++) {
        u128 c = (u128)a.v[0] * b.v[i] + t0;
        const uint64_t lo = (uint64_t)c;
        uint64_t ca = (uint64_t)(c >> 64);
        const uint64_t m = lo * kInv;
        u128 d = (u128)m * kP[0] + lo;
        uint64_t cm = (uint64_t)(d >> 64);
        c = (u128)a.v[1] * b.v[i] + t1 + ca;
        ca = (uint64_t)(c >> 64);
        d = (u128)m * kP[1] + (uint64_t)c + cm;
        t0 = (uint64_t)d;
        cm = (uint64_t)(d >> 64);
        c = (u128)a.v[2] * b.v[i] + t2 + ca;
        ca = (uint64_t)(c >> 64);
        d = (u128)m * kP[2] + (uint64_t)c + cm;
        t1 = (uint64_t)d;
        cm = (uint64_t)(d >> 64);
        c = (u128)a.v[3] * b.v[i] + t3 + ca;
        ca = (uint64_t)(c >> 64);
        d = (u128)m * kP[3] + (uint64_t)c + cm;
        t2 = (uint64_t)d;
        cm = (uint64_t)(d >> 64);
        t3 = cm + ca;
    }
    return cond_sub_p(t0, t1, t2, t3);      // result < 2p
}
inline Fq sqr(const Fq& a) { return mul(a, a); }
inline Fq inv(const Fq& a) {    // a^(p-2)
    uint64_t e[4] = {kP[0] - 2, kP[1], kP[2], kP[3]};
    Fq acc = kOne, base = a;
    for (int i = 0; i < 254; i++) {
        if ((e[i >> 6] >> (i & 63)) & 1) acc = mul(acc, base);
        base = sqr(base);
    }
    return acc;
}
// 32 B little-endian standard form -> Montgomery; false if >= q
inline bool from_std(const uint8_t* b, Fq& out) {
    Fq s;
    memcpy(s.v, b, 32);
    if (geq_p(s.v)) return false;
    out = mul(s, kR2);
    return true;
}
inline Fq from_mont_bytes(const uint8_t* b) {
    Fq s;
    memcpy(s.v, b, 32);
    return s;
}

// ------------------------------------------------------------------------------------------------ Fq2
struct Fq2 {
    Fq c0, c1;
};
const Fq2 kZero2 = {kZero, kZero};
const Fq2 kOne2 = {kOne, kZero};
inline bool is_zero(const Fq2& a) { return is_zero(a.c0) && is_zero(a.c1); }
inline bool eq(const Fq2& a, const Fq2& b) { return eq(a.c0, b.c0) && eq(a.c1, b.c1); }
inline Fq2 add(const Fq2& a, const Fq2& b) { return {add(a.c0, b.c0), add(a.c1, b.c1)}; }
inline Fq2 sub(const Fq2& a, const Fq2& b) { return {sub(a.c0, b.c0), sub(a.c1, b.c1)}; }
inline Fq2 neg(const Fq2& a) { return {neg(a.c0), neg(a.c1)}; }
inline Fq2 dbl(const Fq2& a) { return {dbl(a.c0), dbl(a.c1)}; }
inline Fq2 conj(const Fq2& a) { return {a.c0, neg(a.c1)}; }
inline Fq2 mul(const Fq2& a, const Fq2& b) {
    Fq t0 = mul(a.c0, b.c0), t1 = mul(a.c1, b.c1);
    Fq t2 = mul(add(a.c0, a.c1), add(b.c0, b.c1));
    return {sub(t0, t1), sub(sub(t2, t0), t1)};
}
inline Fq2 sqr(const Fq2& a) {
    Fq t = mul(a.c0, a.c1);
    return {mul(add(a.c0, a.c1), sub(a.c0, a.c1)), dbl(t)};
}
inline Fq2 mul_fq(const Fq2& a, const Fq& k) { return {mul(a.c0, k), mul(a.c1, k)}; }
inline Fq2 inv(const Fq2& a) {
    Fq n = inv(add(sqr(a.c0), sqr(a.c1)));
    return {mul(a.c0, n), neg(mul(a.c1, n))};
}
inline Fq2 mul_xi(const Fq2& a) {    // (9 + u)(c0 + c1 u) = (9 c0 - c1) + (9 c1 + c0) u
    Fq n0 = add(dbl(dbl(dbl(a.c0))), a.c0), n1 = add(dbl(dbl(dbl(a.c1))), a.c1);
    return {sub(n0, a.c1), add(n1, a.c0)};
}
inline Fq2 fq2_from_u64(const uint64_t (*c)[4]) {
    Fq2 r;
    memcpy(r.c0.v, c[0], 32);
    memcpy(r.c1.v, c[1], 32);
    return r;
}

// gamma[k-1][i-1] = xi^(i (q^k - 1)/6), Montgomery form (generated with the oracle's Fq2 arithmetic;
// cross-checked by tests/test_verify.py through Frobenius consistency of the pairing itself)
const uint64_t kGamma[3][5][2][4] = {
    {
        {{0xaf9ba69633144907ull, 0xca6b1d7387afb78aull, 0x11bded5ef08a2087ull, 0x02f34d751a1f3a7cull},
         {0xa222ae234c492d72ull, 0xd00f02a4565de15bull, 0xdc2ff3a253dfc926ull, 0x10a75716b3899551ull}},
        {{0xb5773b104563ab30ull, 0x347f91c8a9aa6454ull, 0x7a007127242e0991ull, 0x1956bcd8118214ecull},
         {0x6e849f1ea0aa4757ull, 0xaa1c7b6d89f89141ull, 0xb6e713cdfae0ca3aull, 0x26694fbb4e82ebc3ull}},
        {{0xe4bbdd0c2936b629ull, 0xbb30f162e133bacbull, 0x31a9d1b6f9645366ull, 0x253570bea500f8ddull},
         {0xa1d77ce45ffe77c7ull, 0x07affd117826d1dbull, 0x6d16bd27bb7edc6bull, 0x2c87200285defeccull}},
        {{0x7361d77f843abe92ull, 0xa5bb2bd3273411fbull, 0x9c941f314b3e2399ull, 0x15df9cddbb9fd3ecull},
         {0x5dddfd154bd8c949ull, 0x62cb29a5a4445b60ull, 0x37bc870a0c7dd2b9ull, 0x24830a9d3171f0fdull}},
        {{0xc970692f41690fe7ull, 0xe240342127694b0bull, 0x32bee66b83c459e8ull, 0x12aabced0ab08841ull},
         {0x0d485d2340aebfa9ull, 0x05193418ab2fcc57ull, 0xd3b0a40b8a4910f5ull, 0x2f21ebb535d2925aull}},
    },
    {
        {{0xca8d800500fa1bf2ull, 0xf0c5d61468b39769ull, 0x0e201271ad0d4418ull, 0x04290f65bad856e6ull}, {0, 0, 0, 0}},
        {{0x3350c88e13e80b9cull, 0x7dce557cdb5e56b9ull, 0x6001b4b8b615564aull, 0x2682e617020217e0ull}, {0, 0, 0, 0}},
        {{0x68c3488912edefaaull, 0x8d087f6872aabf4full, 0x51e1a24709081231ull, 0x2259d6b14729c0faull}, {0, 0, 0, 0}},
        {{0x71930c11d782e155ull, 0xa6bb947cffbe3323ull, 0xaa303344d4741444ull, 0x2c3b3f0d26594943ull}, {0, 0, 0, 0}},
        {{0x08cfc388c494f1abull, 0x19b315148d1373d4ull, 0x584e90fdcb6c0213ull, 0x09e1685bdf2f8849ull}, {0, 0, 0, 0}},
    },
    {
        {{0x365316184e46d97dull, 0x0af7129ed4c96d9full, 0x659da72fca1009b5ull, 0x08116d8983a20d23ull},
         {0xb1df4af7c39c1939ull, 0x3d9f02878a73bf7full, 0x9b2220928caf0ae0ull, 0x26684515eff054a6ull}},
        {{0xc9af22f716ad6badull, 0xb311782a4aa662b2ull, 0x19eeaf64e248c7f4ull, 0x20273e77e3439f82ull},
         {0xacc02860f7ce93acull, 0x3933d5817ba76b4cull, 0x69e6188b446c8467ull, 0x0a46036d4417cc55ull}},
        {{0x5764af0aaf46471eull, 0xdc50792e873e0fc1ull, 0x86a673ff881d04f6ull, 0x0b2eddb43c30a74cull},
         {0x9a490f32787e8580ull, 0x8fd16d7ff04af8b1ull, 0x4b39888ec6027bf2ull, 0x03dd2e705b52a15dull}},
        {{0x448a93a57b6762dfull, 0xbfd62df528fdeadfull, 0xd858f5d00e9bd47aull, 0x06b03d4d3476ec58ull},
         {0x2b19daf4bcc936d1ull, 0xa1a54e7a56f4299full, 0xb533eee05adeaef1ull, 0x170c812b84dda0b2ull}},
        {{0xe0bc4b2275cf559full, 0xc238b945c154e60full, 0x803982a5929a7d5eull, 0x15ce052df7e4a37eull},
         {0x2d28efbdbf3799a7ull, 0x9b097e3c1ad60773ull, 0x982d4113af4a535bull, 0x24e18991e3056063ull}},
    },
};
// twist coefficient b' = 3 / (9 + u), Montgomery (TxVerifier.sol's precompile curve: y^2 = x^3 + 3/(9+u))
const uint64_t kTwistB[2][4] = {{0x3bf938e377b802a8ull, 0x020b1b273633535dull, 0x26b7edf049755260ull, 0x2514c6324384a86dull},
                                {0x38e7ecccd1dcff67ull, 0x65f0b37d93ce0d3eull, 0xd749d0dd22ac00aaull, 0x0141b9ce4a688d4dull}};
const Fq kThree = {{0x7a17caa950ad28d7ull, 0x1f6ac17ae15521b9ull, 0x334bea4e696bd284ull, 0x2a1f6744ce179d8eull}};
const uint64_t kBnX = 4965661367192848881ull;                         // BN parameter x
const u128 kAteLoop = ((u128)0x1ull << 64) | 0x9d797039be763ba8ull;   // 6x + 2 = 29793968203157093288 (65 bits)

inline Fq2 gamma(int k, int i) { return fq2_from_u64(kGamma[k - 1][i - 1]); }

// ------------------------------------------------------------------------------------------------ Fq12
struct Fq12 {
    Fq2 c[6];      // sum c[i] w^i, w^6 = xi
};
inline Fq12 f12_one() {
    Fq12 r;
    r.c[0] = kOne2;
    for (int i = 1; i < 6; i++) r.c[i] = kZero2;
    return r;
}
inline bool f12_is_one(const Fq12& a) {
    if (!eq(a.c[0], kOne2)) return false;
    for (int i = 1; i < 6; i++)
        if (!is_zero(a.c[i])) return false;
    return true;
}
// (a0 + a1 x + a2 x^2)(b0 + b1 x + b2 x^2) -> c[0..4], 6 Fq2 multiplications (Karatsuba)
inline void poly3_mul(const Fq2* a, const Fq2* b, Fq2* c) {
    Fq2 v0 = mul(a[0], b[0]), v1 = mul(a[1], b[1]), v2 = mul(a[2], b[2]);
    c[0] = v0;
    c[1] = sub(sub(mul(add(a[0], a[1]), add(b[0], b[1])), v0), v1);
    c[2] = add(sub(sub(mul(add(a[0], a[2]), add(b[0], b[2])), v0), v2), v1);
    c[3] = sub(sub(mul(add(a[1], a[2]), add(b[1], b[2])), v1), v2);
    c[4] = v2;
}
// a = P0 + P1 w^3, b = Q0 + Q1 w^3 (halves of degree < 3 in w): Karatsuba over the halves, 18 Fq2 multiplications
Fq12 f12_mul(const Fq12& a, const Fq12& b) {
    Fq2 lo[5], hi[5], mid[5], sa[3], sb[3];
    poly3_mul(a.c, b.c, lo);
    poly3_mul(a.c + 3, b.c + 3, hi);
    for (int i = 0; i < 3; i++) {
        sa[i] = add(a.c[i], a.c[i + 3]);
        sb[i] = add(b.c[i], b.c[i + 3]);
    }
    poly3_mul(sa, sb, mid);
    Fq2 t[11];
    for (int i = 0; i < 11; i++) t[i] = kZero2;
    for (int i = 0; i < 5; i++) {
        t[i] = add(t[i], lo[i]);
        t[i + 3] = add(t[i + 3], sub(sub(mid[i], lo[i]), hi[i]));
        t[i + 6] = add(t[i + 6], hi[i]);
    }
    Fq12 r;
    for (int k = 0; k < 6; k++) r.c[k] = k < 5 ? add(t[k], mul_xi(t[k + 6])) : t[k];
    return r;
}
// Squaring over the quadratic tower Fq12 = Fq6[w]/(w^2 - v), Fq6 = Fq2[v]/(v^3 - xi), v = w^2: with a = E + O w
// (E = c0 + c2 v + c4 v^2, O = c1 + c3 v + c5 v^2),  a^2 = (E^2 + v O^2) + 2 E O w  and
// E^2 + v O^2 = (E + O)(E + v O) - E O - v E O: two Fq6 products (12 Fq2 multiplications) instead of 18.
inline void f6_mul(const Fq2* a, const Fq2* b, Fq2* r) {      // in Fq2[v]/(v^3 - xi)
    Fq2 c[5];
    poly3_mul(a, b, c);
    r[0] = add(c[0], mul_xi(c[3]));
    r[1] = add(c[1], mul_xi(c[4]));
    r[2] = c[2];
}
Fq12 f12_sqr(const Fq12& a) {
    const Fq2 E[3] = {a.c[0], a.c[2], a.c[4]}, O[3] = {a.c[1], a.c[3], a.c[5]};
    const Fq2 vO[3] = {mul_xi(O[2]), O[0], O[1]};             // v * O
    const Fq2 s1[3] = {add(E[0], O[0]), add(E[1], O[1]), add(E[2], O[2])};
    const Fq2 s2[3] = {add(E[0], vO[0]), add(E[1], vO[1]), add(E[2], vO[2])};
    Fq2 eo[3], m[3];
    f6_mul(E, O, eo);
    f6_mul(s1, s2, m);
    const Fq2 veo[3] = {mul_xi(eo[2]), eo[0], eo[1]};
    Fq12 r;
    for (int i = 0; i < 3; i++) {
        r.c[2 * i] = sub(sub(m[i], eo[i]), veo[i]);
        r.c[2 * i + 1] = dbl(eo[i]);
    }
    return r;
}
// a * (l0 + l1 w + l3 w^3), l0 in Fq
Fq12 f12_mul_line(const Fq12& a, const Fq& l0, const Fq2& l1, const Fq2& l3) {
    Fq2 t[9];
    for (int i = 0; i < 9; i++) t[i] = kZero2;
    for (int i = 0; i < 6; i++) {
        t[i] = add(t[i], mul_fq(a.c[i], l0));
        t[i + 1] = add(t[i + 1], mul(a.c[i], l1));
        t[i + 3] = add(t[i + 3], mul(a.c[i], l3));
    }
    Fq12 r;
    for (int k = 0; k < 6; k++) r.c[k] = k < 3 ? add(t[k], mul_xi(t[k + 6])) : t[k];
    return r;
}
// a * (l0 + l1 w + l3 w^3), l0 in Fq2 (projective Miller loop: the line is scaled by an Fq2 factor, which the
// final exponentiation removes).  Schoolbook version: 18 Fq2 multiplications; kept as the self-check reference.
Fq12 f12_mul_line2_ref(const Fq12& a, const Fq2& l0, const Fq2& l1, const Fq2& l3) {
    Fq2 t[9];
    for (int i = 0; i < 9; i++) t[i] = kZero2;
    for (int i = 0; i < 6; i++) {
        t[i] = add(t[i], mul(a.c[i], l0));
        t[i + 1] = add(t[i + 1], mul(a.c[i], l1));
        t[i + 3] = add(t[i + 3], mul(a.c[i], l3));
    }
    Fq12 r;
    for (int k = 0; k < 6; k++) r.c[k] = k < 3 ? add(t[k], mul_xi(t[k + 6])) : t[k];
    return r;
}
// (a0 + a1 v + a2 v^2)(x0 + x1 v) in Fq2[v]/(v^3 - xi): 5 Fq2 multiplications
inline void f6_mul_by_01(const Fq2* a, const Fq2& x0, const Fq2& x1, Fq2* r) {
    const Fq2 t0 = mul(a[0], x0), t1 = mul(a[1], x1);
    r[1] = sub(sub(mul(add(a[0], a[1]), add(x0, x1)), t0), t1);
    r[0] = add(t0, mul_xi(mul(a[2], x1)));
    r[2] = add(t1, mul(a[2], x0));
}
// Same product over the tower (v = w^2): a = E + O w, line = L0 + L1 w with L0 = l0, L1 = l1 + l3 v;
//   a * line = (E L0 + v O L1) + ((E + O)(L0 + L1) - E L0 - O L1) w :  3 + 5 + 5 = 13 Fq2 multiplications.
Fq12 f12_mul_line2(const Fq12& a, const Fq2& l0, const Fq2& l1, const Fq2& l3) {
    const Fq2 E[3] = {a.c[0], a.c[2], a.c[4]}, O[3] = {a.c[1], a.c[3], a.c[5]};
    const Fq2 S[3] = {add(E[0], O[0]), add(E[1], O[1]), add(E[2], O[2])};
    Fq2 t0[3], t1[3], t2[3];
    for (int i = 0; i < 3; i++) t0[i] = mul(E[i], l0);
    f6_mul_by_01(O, l1, l3, t1);
    f6_mul_by_01(S, add(l0, l1), l3, t2);
    const Fq2 vt1[3] = {mul_xi(t1[2]), t1[0], t1[1]};
    Fq12 r;
    for (int i = 0; i < 3; i++) {
        r.c[2 * i] = add(t0[i], vt1[i]);
        r.c[2 * i + 1] = sub(sub(t2[i], t0[i]), t1[i]);
    }
    static const bool self_check = getenv("ZKR_PAIRING_CYC") && atoi(getenv("ZKR_PAIRING_CYC")) == 2;
    if (self_check) {
        const Fq12 g = f12_mul_line2_ref(a, l0, l1, l3);
        for (int k = 0; k < 6; k++)
            if (!eq(g.c[k], r.c[k])) {
                fprintf(stderr, "zkr: sparse line product self-check FAILED\n");
                abort();
            }
    }
    return r;
}
inline Fq12 f12_conj(const Fq12& a) {       // the q^6 Frobenius: w -> -w
    Fq12 r = a;
    r.c[1] = neg(a.c[1]);
    r.c[3] = neg(a.c[3]);
    r.c[5] = neg(a.c[5]);
    return r;
}
// a^(q^k), k = 1, 2, 3:  (c_i w^i)^(q^k) = conj^k(c_i) gamma_k^i w^i
Fq12 f12_frob(const Fq12& a, int k) {
    Fq12 r;
    for (int i = 0; i < 6; i++) {
        Fq2 c = (k & 1) ? conj(a.c[i]) : a.c[i];
        r.c[i] = i == 0 ? c : mul(c, gamma(k, i));
    }
    return r;
}
// inverse through the norm to Fq:  a^-1 = a^(q + q^2 + ... + q^11) / N(a)
Fq12 f12_inv(const Fq12& a) {
    Fq12 s1 = f12_frob(a, 1);                                    // a^q
    Fq12 s2 = f12_mul(s1, f12_frob(s1, 1));                      // a^(q + q^2)
    Fq12 s3 = f12_mul(s2, f12_frob(s1, 2));                      // a^(q + q^2 + q^3)
    Fq12 s4 = f12_mul(s2, f12_frob(s2, 2));                      // a^(q + .. + q^4)
    Fq12 s8 = f12_mul(s4, f12_frob(f12_frob(s4, 2), 2));         // a^(q + .. + q^8)
    Fq12 t = s3;
    for (int i = 0; i < 4; i++) t = f12_frob(t, 2);              // a^(q^9 + q^10 + q^11)
    Fq12 rr = f12_mul(s8, t);                                    // a^(q + .. + q^11)
    Fq12 n = f12_mul(a, rr);                                     // norm, lies in Fq
    Fq ninv = inv(n.c[0].c0);
    Fq12 out;
    for (int i = 0; i < 6; i++) out.c[i] = mul_fq(rr.c[i], ninv);
    return out;
}
// Squaring in the cyclotomic subgroup G_{Phi_6(q^2)} (every value after the easy part of the final exponentiation):
// Granger, Scott, "Faster squaring in the cyclotomic subgroup of sixth degree extensions".  View Fq12 as
// Fq4[w]/(w^3 - s), Fq4 = Fq2[s]/(s^2 - xi), s = w^3:  a = A + B w + C w^2 with A = c0 + c3 s, B = c1 + c4 s, C = c2 + c5 s;
//   a^2 = (3 A^2 - 2 conj(A)) + (3 s C^2 + 2 conj(B)) w + (3 B^2 - 2 conj(C)) w^2,   conj(x0 + x1 s) = x0 - x1 s.
// 3 Fq4 squarings = 9 Fq2 squarings instead of the 12 Fq2 multiplications of f12_sqr.
inline void f4_sqr(const Fq2& x0, const Fq2& x1, Fq2& y0, Fq2& y1) {
    const Fq2 a = sqr(x0), b = sqr(x1);
    y1 = sub(sub(sqr(add(x0, x1)), a), b);
    y0 = add(a, mul_xi(b));
}
inline Fq2 triple(const Fq2& a) { return add(dbl(a), a); }
Fq12 f12_cyc_sqr(const Fq12& a) {
    Fq2 a0, a1, b0, b1, c0, c1;
    f4_sqr(a.c[0], a.c[3], a0, a1);       // A^2
    f4_sqr(a.c[1], a.c[4], b0, b1);       // B^2
    f4_sqr(a.c[2], a.c[5], c0, c1);       // C^2,  s C^2 = xi c1 + c0 s
    Fq12 r;
    r.c[0] = sub(triple(a0), dbl(a.c[0]));
    r.c[3] = add(triple(a1), dbl(a.c[3]));
    r.c[1] = add(triple(mul_xi(c1)), dbl(a.c[1]));
    r.c[4] = sub(triple(c0), dbl(a.c[4]));
    r.c[2] = sub(triple(b0), dbl(a.c[2]));
    r.c[5] = add(triple(b1), dbl(a.c[5]));
    return r;
}
// a^x for a in the cyclotomic subgroup
Fq12 f12_exp_x(const Fq12& a) {
    static const int mode = getenv("ZKR_PAIRING_CYC") ? atoi(getenv("ZKR_PAIRING_CYC")) : 1;   // 0: generic squarings, 2: self-check
    Fq12 r = a;
    for (int i = 61; i >= 0; i--) {       // kBnX has 63 bits, top bit consumed by r = a
        if (mode == 2) {
            const Fq12 g = f12_sqr(r), c = f12_cyc_sqr(r);
            for (int k = 0; k < 6; k++)
                if (!eq(g.c[k], c.c[k])) {
                    fprintf(stderr, "zkr: cyclotomic squaring self-check FAILED\n");
                    abort();
                }
            r = c;
        } else {
            r = mode ? f12_cyc_sqr(r) : f12_sqr(r);
        }
        if ((kBnX >> i) & 1) r = f12_mul(r, a);
    }
    return r;
}
// f^((q^12 - 1) / r): easy part (q^6 - 1)(q^2 + 1), hard part of Scott, Benger, Charlemagne, Dominguez Perez,
// Kachisa, "On the final exponentiation for calculating pairings on ordinary elliptic curves" (BN case)
Fq12 final_exp(const Fq12& in) {
    Fq12 t1 = f12_mul(f12_conj(in), f12_inv(in));
    t1 = f12_mul(f12_frob(t1, 2), t1);
    Fq12 fp = f12_frob(t1, 1), fp2 = f12_frob(t1, 2), fp3 = f12_frob(fp2, 1);
    Fq12 fu = f12_exp_x(t1), fu2 = f12_exp_x(fu), fu3 = f12_exp_x(fu2);
    Fq12 y3 = f12_conj(f12_frob(fu, 1));
    Fq12 fu2p = f12_frob(fu2, 1), fu3p = f12_frob(fu3, 1);
    Fq12 y2 = f12_frob(fu2, 2);
    Fq12 y0 = f12_mul(f12_mul(fp, fp2), fp3);
    Fq12 y1 = f12_conj(t1);
    Fq12 y5 = f12_conj(fu2);
    Fq12 y4 = f12_conj(f12_mul(fu, fu2p));
    Fq12 y6 = f12_conj(f12_mul(fu3, fu3p));
    Fq12 t0 = f12_mul(f12_mul(f12_sqr(y6), y4), y5);
    Fq12 u1 = f12_mul(f12_mul(y3, y5), t0);
    t0 = f12_mul(t0, y2);
    u1 = f12_sqr(f12_mul(f12_sqr(u1), t0));
    t0 = f12_mul(u1, y1);
    u1 = f12_mul(u1, y0);
    t0 = f12_sqr(t0);
    return f12_mul(t0, u1);
}

// ------------------------------------------------------------------------------------------------ curves
struct G1A {
    Fq x, y;
    bool inf;
};
struct G2A {
    Fq2 x, y;
    bool inf;
};
inline bool on_curve(const G1A& p) { return p.inf || eq(sqr(p.y), add(mul(sqr(p.x), p.x), kThree)); }
inline bool on_curve(const G2A& p) {
    return p.inf || eq(sqr(p.y), add(mul(sqr(p.x), p.x), fq2_from_u64(kTwistB)));
}

// Jacobian arithmetic, generic over Fq / Fq2 (only for the subgroup check and vk_x = IC[0] + msm)
template <class F>
struct Jac {
    F x, y, z;
    bool inf;
};
template <class F>
Jac<F> jdbl(const Jac<F>& p) {
    if (p.inf || is_zero(p.y)) return {p.x, p.y, p.z, true};
    F a = sqr(p.x), b = sqr(p.y), c = sqr(b);
    F d = dbl(sub(sub(sqr(add(p.x, b)), a), c));
    F e = add(dbl(a), a), f = sqr(e);
    F x3 = sub(f, dbl(d));
    F y3 = sub(mul(e, sub(d, x3)), dbl(dbl(dbl(c))));
    F z3 = dbl(mul(p.y, p.z));
    return {x3, y3, z3, false};
}
template <class F>
Jac<F> jadd_affine(const Jac<F>& p, const F& qx, const F& qy, const F& one) {
    if (p.inf) return {qx, qy, one, false};
    F z1z1 = sqr(p.z);
    F u2 = mul(qx, z1z1), s2 = mul(mul(qy, p.z), z1z1);
    F h = sub(u2, p.x), rr = sub(s2, p.y);
    if (is_zero(h)) {
        if (is_zero(rr)) return jdbl(p);
        return {p.x, p.y, p.z, true};
    }
    F hh = sqr(h), hhh = mul(h, hh), v = mul(p.x, hh);
    F x3 = sub(sub(sqr(rr), hhh), dbl(v));
    F y3 = sub(mul(rr, sub(v, x3)), mul(p.y, hhh));
    F z3 = mul(p.z, h);
    return {x3, y3, z3, false};
}
// [r] Q == O ?   (the alt_bn128 pairing precompile rejects G2 points outside the order-r subgroup)
bool g2_in_subgroup(const G2A& q) {
    if (q.inf) return true;
    Jac<Fq2> acc = {q.x, q.y, kOne2, true};
    for (int i = 253; i >= 0; i--) {
        acc = jdbl(acc);
        if ((kRmod[i >> 6] >> (i & 63)) & 1) acc = jadd_affine(acc, q.x, q.y, kOne2);
    }
    return acc.inf;
}
G1A g1_add(const G1A& a, const G1A& b) {
    if (a.inf) return b;
    if (b.inf) return a;
    Jac<Fq> j = jadd_affine<Fq>({a.x, a.y, kOne, false}, b.x, b.y, kOne);
    if (j.inf) return {kZero, kZero, true};
    Fq zi = inv(j.z), zi2 = sqr(zi);
    return {mul(j.x, zi2), mul(j.y, mul(zi2, zi)), false};
}

// ------------------------------------------------------------------------------------------------ pairing
struct MillerState {
    Fq2 tx, ty;        // running twist point T (affine)
    Fq2 qx, qy;        // Q
    Fq px, py;         // P
};

// batch inversion (Montgomery's trick); returns false if some element is zero
bool batch_inv(Fq2* d, int n) {
    if (n == 0) return true;
    Fq2 pref[8];
    Fq2 acc = kOne2;
    for (int i = 0; i < n; i++) {
        if (is_zero(d[i])) return false;
        pref[i] = acc;
        acc = mul(acc, d[i]);
    }
    Fq2 ia = inv(acc);
    for (int i = n - 1; i >= 0; i--) {
        Fq2 di = mul(ia, pref[i]);
        ia = mul(ia, d[i]);
        d[i] = di;
    }
    return true;
}

// one line step for every pair: T <- T + S (S = T for a doubling, else the given point), f <- f * l_{T,S}(P).
// Untwist psi(x, y) = (x w^2, y w^3):  l(P) = yP - lambda xP w + (lambda x1 - y1) w^3.
bool line_step(Fq12& f, MillerState* st, int n, bool doubling, const Fq2* sx, const Fq2* sy) {
    Fq2 den[8];
    for (int i = 0; i < n; i++) den[i] = doubling ? dbl(st[i].ty) : sub(sx[i], st[i].tx);
    if (!batch_inv(den, n)) return false;       // cannot happen for points of order r (see header of zkr_pairing_check)
    for (int i = 0; i < n; i++) {
        MillerState& s = st[i];
        Fq2 lam;
        if (doubling) {
            Fq2 x2 = sqr(s.tx);
            lam = mul(add(dbl(x2), x2), den[i]);
        } else {
            lam = mul(sub(sy[i], s.ty), den[i]);
        }
        const Fq2& ox = doubling ? s.tx : sx[i];
        Fq2 x3 = sub(sub(sqr(lam), s.tx), ox);
        Fq2 y3 = sub(mul(lam, sub(s.tx, x3)), s.ty);
        Fq2 l1 = neg(mul_fq(lam, s.px));
        Fq2 l3 = sub(mul(lam, s.tx), s.ty);
        f = f12_mul_line(f, s.py, l1, l3);
        s.tx = x3;
        s.ty = y3;
    }
    return true;
}

// ---- the same loop in homogeneous projective coordinates: no inversion at all (the affine loop above pays one Fq
// inversion = ~380 multiplications per line step, which is most of its time for a 4-pair product).
// Formulas of Costello, Lange, Naehrig, "Faster pairing computations on curves with high-degree twists" (D-type twist
// y^2 = x^3 + b'), lines scaled by an element of Fq2:
//   doubling   T = (X, Y, Z):  l = -2YZ yP + 3X^2 xP w + (3b'Z^2 - Y^2) w^3
//   addition   T + Q, Q affine: theta = Y - yQ Z, lambda = X - xQ Z:  l = lambda yP - theta xP w + (theta xQ - lambda yQ) w^3
// (the affine lines yP - lam xP w + (lam x1 - y1) w^3 times -2YZ, resp. times lambda).
struct ProjState {
    Fq2 x, y, z;       // running twist point T
    Fq2 qx, qy;        // Q
    Fq px, py;         // P
};
inline Fq half(const Fq& a) {                 // a / 2 mod p
    static const Fq kHalf = inv(add(kOne, kOne));
    return mul(a, kHalf);
}
inline Fq2 half(const Fq2& a) { return {half(a.c0), half(a.c1)}; }
inline void proj_double_step(Fq12& f, ProjState& s) {
    const Fq2 bt = fq2_from_u64(kTwistB);
    Fq2 a = half(mul(s.x, s.y));
    Fq2 b = sqr(s.y), c = sqr(s.z);
    Fq2 e = mul(bt, add(dbl(c), c));
    Fq2 ff = add(dbl(e), e);
    Fq2 g = half(add(b, ff));
    Fq2 h = sub(sqr(add(s.y, s.z)), add(b, c));
    Fq2 i = sub(e, b);
    Fq2 j = sqr(s.x);
    Fq2 e2 = sqr(e);
    s.x = mul(a, sub(b, ff));
    s.y = sub(sqr(g), add(dbl(e2), e2));
    s.z = mul(b, h);
    f = f12_mul_line2(f, neg(mul_fq(h, s.py)), mul_fq(add(dbl(j), j), s.px), i);
}
// false: T == +-S (cannot happen for points of order r inside the loop)
inline bool proj_add_step(Fq12& f, ProjState& s, const Fq2& sx, const Fq2& sy) {
    Fq2 theta = sub(s.y, mul(sy, s.z));
    Fq2 lambda = sub(s.x, mul(sx, s.z));
    if (is_zero(lambda)) return false;
    Fq2 c = sqr(theta), d = sqr(lambda);
    Fq2 e = mul(lambda, d), ff = mul(s.z, c), g = mul(s.x, d);
    Fq2 h = sub(add(e, ff), dbl(g));
    Fq2 y3 = sub(mul(theta, sub(g, h)), mul(e, s.y));
    s.x = mul(lambda, h);
    s.y = y3;
    s.z = mul(s.z, e);
    Fq2 j = sub(mul(theta, sx), mul(lambda, sy));
    f = f12_mul_line2(f, mul_fq(lambda, s.py), neg(mul_fq(theta, s.px)), j);
    return true;
}
bool miller_product_projective(const G1A* P, const G2A* Q, int n_in, Fq12* out) {
    ProjState st[8];
    int n = 0;
    for (int i = 0; i < n_in; i++) {
        if (P[i].inf || Q[i].inf) continue;       // e(O, Q) = e(P, O) = 1
        st[n++] = {Q[i].x, Q[i].y, kOne2, Q[i].x, Q[i].y, P[i].x, P[i].y};
    }
    Fq12 f = f12_one();
    if (n) {
        for (int b = 63; b >= 0; b--) {           // bits below the leading one of the 65-bit loop count
            f = f12_sqr(f);
            for (int i = 0; i < n; i++) {
                if (is_zero(st[i].y)) return false;
                proj_double_step(f, st[i]);
            }
            if ((kAteLoop >> b) & 1)
                for (int i = 0; i < n; i++)
                    if (!proj_add_step(f, st[i], st[i].qx, st[i].qy)) return false;
        }
        // Q1 = pi(Q), -Q2 = -pi^2(Q) on the twist
        const Fq2 g12 = gamma(1, 2), g13 = gamma(1, 3), g22 = gamma(2, 2), g23 = gamma(2, 3);
        for (int i = 0; i < n; i++) {
            if (!proj_add_step(f, st[i], mul(conj(st[i].qx), g12), mul(conj(st[i].qy), g13))) return false;
            if (!proj_add_step(f, st[i], mul(st[i].qx, g22), neg(mul(st[i].qy, g23)))) return false;
        }
    }
    *out = f;
    return true;
}

// prod_i e(P_i, Q_i) == 1 ?   ok=false: a degenerate line was hit (inputs outside the prime-order groups)
bool pairing_product_is_one_affine(const G1A* P, const G2A* Q, int n_in, bool* ok);
bool pairing_product_is_one(const G1A* P, const G2A* Q, int n_in, bool* ok) {
    static const bool use_affine = getenv("ZKR_PAIRING_AFFINE") && atoi(getenv("ZKR_PAIRING_AFFINE"));   // cross-check knob
    if (use_affine) return pairing_product_is_one_affine(P, Q, n_in, ok);
    Fq12 f;
    *ok = miller_product_projective(P, Q, n_in, &f);
    if (!*ok) return false;
    return f12_is_one(final_exp(f));
}
bool pairing_product_is_one_affine(const G1A* P, const G2A* Q, int n_in, bool* ok) {
    MillerState st[8];
    int n = 0;
    for (int i = 0; i < n_in; i++) {
        if (P[i].inf || Q[i].inf) continue;       // e(O, Q) = e(P, O) = 1
        st[n++] = {Q[i].x, Q[i].y, Q[i].x, Q[i].y, P[i].x, P[i].y};
    }
    *ok = true;
    Fq12 f = f12_one();
    if (n) {
        Fq2 qx[8], qy[8];
        for (int i = 0; i < n; i++) {
            qx[i] = st[i].qx;
            qy[i] = st[i].qy;
        }
        for (int b = 63; b >= 0; b--) {           // bits below the leading one of the 65-bit loop count
            f = f12_sqr(f);
            if (!line_step(f, st, n, true, nullptr, nullptr)) return *ok = false;
            if ((kAteLoop >> b) & 1)
                if (!line_step(f, st, n, false, qx, qy)) return *ok = false;
        }
        // Q1 = pi(Q), -Q2 = -pi^2(Q) on the twist
        Fq2 g12 = gamma(1, 2), g13 = gamma(1, 3), g22 = gamma(2, 2), g23 = gamma(2, 3);
        Fq2 ax[8], ay[8];
        for (int i = 0; i < n; i++) {
            ax[i] = mul(conj(qx[i]), g12);
            ay[i] = mul(conj(qy[i]), g13);
        }
        if (!line_step(f, st, n, false, ax, ay)) return *ok = false;
        for (int i = 0; i < n; i++) {
            ax[i] = mul(qx[i], g22);
            ay[i] = neg(mul(qy[i], g23));
        }
        if (!line_step(f, st, n, false, ax, ay)) return *ok = false;
    }
    return f12_is_one(final_exp(f));
}

// ------------------------------------------------------------------------------------------------ decoding
// x|y standard form, all-zero = infinity (zkr.h proof encoding; also the EVM's encoding of the zero point)
bool g1_from_std(const uint8_t* b, G1A& p) {
    bool z = true;
    for (int i = 0; i < 64; i++) z &= b[i] == 0;
    if (z) {
        p = {kZero, kZero, true};
        return true;
    }
    p.inf = false;
    return from_std(b, p.x) && from_std(b + 32, p.y);
}
bool g2_from_std(const uint8_t* b, G2A& p) {
    bool z = true;
    for (int i = 0; i < 128; i++) z &= b[i] == 0;
    if (z) {
        p = {kZero2, kZero2, true};
        return true;
    }
    p.inf = false;
    return from_std(b, p.x.c0) && from_std(b + 32, p.x.c1) && from_std(b + 64, p.y.c0) && from_std(b + 96, p.y.c1);
}
// Montgomery bytes (binary key encoding); x == 0 marks infinity (binarify.ts:92-95 drops z)
G1A g1_from_mont(const uint8_t* b) {
    G1A p = {from_mont_bytes(b), from_mont_bytes(b + 32), false};
    p.inf = is_zero(p.x);
    return p;
}
G2A g2_from_mont(const uint8_t* b) {
    G2A p = {{from_mont_bytes(b), from_mont_bytes(b + 32)}, {from_mont_bytes(b + 64), from_mont_bytes(b + 96)}, false};
    p.inf = is_zero(p.x);
    return p;
}

}  // namespace pr

// ---- host_ec.cuh: byte-level checks and pairings for the setup ceremony (ceremony.cu)
int host_point_check(int group, const void* mont, bool subgroup) {
    const uint8_t* b = (const uint8_t*)mont;
    const int coords = group == 1 ? 2 : 4;
    bool xz = true;
    for (int i = 0; i < 16 * coords; i++) xz &= b[i] == 0;
    if (xz) return PT_INFINITY;
    for (int i = 0; i < coords; i++) {
        uint64_t v[4];
        memcpy(v, b + 32 * i, 32);
        if (pr::geq_p(v)) return PT_RANGE;
    }
    if (group == 1) return pr::on_curve(pr::g1_from_mont(b)) ? PT_OK : PT_OFF_CURVE;
    const pr::G2A q = pr::g2_from_mont(b);
    if (!pr::on_curve(q)) return PT_OFF_CURVE;
    return !subgroup || pr::g2_in_subgroup(q) ? PT_OK : PT_SUBGROUP;
}

bool host_pairing_is_one(const void* const* g1_mont, const bool* negate, const void* const* g2_mont, int n) {
    pr::G1A P[8];
    pr::G2A Q[8];
    for (int i = 0; i < n; i++) {
        P[i] = pr::g1_from_mont((const uint8_t*)g1_mont[i]);
        if (negate[i] && !P[i].inf) P[i].y = pr::neg(P[i].y);
        Q[i] = pr::g2_from_mont((const uint8_t*)g2_mont[i]);
    }
    bool ok = true;
    const bool one = pr::pairing_product_is_one(P, Q, n, &ok);
    return ok && one;
}

bool host_g1_std_to_mont(const void* std64, void* mont64) {
    pr::G1A p;
    if (!pr::g1_from_std((const uint8_t*)std64, p)) return false;
    memcpy(mont64, p.inf ? pr::kZero.v : p.x.v, 32);
    memcpy((uint8_t*)mont64 + 32, p.inf ? pr::kZero.v : p.y.v, 32);
    return true;
}

}  // namespace zkr

using namespace zkr;

struct zkr_vkey {
    zkr_ctx* ctx = nullptr;
    uint32_t n_public = 0;
    pr::G1A ic0, alfa1;
    pr::G2A beta2, gamma2, delta2;
    zkr_bases* ic_bases = nullptr;      // IC[1..n_public], window tables resident in HBM
};

static int vkey_finish(zkr_ctx* ctx, const VKeyRaw& raw, zkr_vkey** out) {
    zkr_vkey* vk = new zkr_vkey();
    vk->ctx = ctx;
    vk->n_public = raw.n_public;
    vk->alfa1 = pr::g1_from_mont(raw.alfa1);
    vk->beta2 = pr::g2_from_mont(raw.beta2);
    vk->gamma2 = pr::g2_from_mont(raw.gamma2);
    vk->delta2 = pr::g2_from_mont(raw.delta2);
    vk->ic0 = pr::g1_from_mont(raw.ic.data());
    bool good = pr::on_curve(vk->alfa1) && pr::on_curve(vk->ic0);
    for (uint32_t i = 1; good && i <= raw.n_public; i++) good = pr::on_curve(pr::g1_from_mont(raw.ic.data() + 64 * (size_t)i));
    const pr::G2A* g2s[3] = {&vk->beta2, &vk->gamma2, &vk->delta2};
    for (int i = 0; good && i < 3; i++) good = pr::on_curve(*g2s[i]) && pr::g2_in_subgroup(*g2s[i]);
    if (!good) {
        delete vk;
        set_error("verification key: a point is not on the curve / not in the order-r subgroup");
        return ZKR_E_BADKEY;
    }
    if (raw.n_public) {
        int rc = zkr_bases_load(ctx, 1, raw.ic.data() + 64, raw.n_public, 0, &vk->ic_bases);
        if (rc != ZKR_OK) {
            delete vk;
            return rc;
        }
    }
    *out = vk;
    return ZKR_OK;
}

extern "C" int zkr_vkey_load_json(zkr_ctx* ctx, const char* json, size_t len, zkr_vkey** out) {
    if (!ctx || !json || !out) {
        set_error("zkr_vkey_load_json: null argument");
        return ZKR_E_INVALID;
    }
    *out = nullptr;
    VKeyRaw raw;
    ZKR_TRY(vkey_parse_json(json, len, &raw));
    return vkey_finish(ctx, raw, out);
}

// buf: alfa1 | beta1 | delta1 (64 B each) | beta2 | gamma2 | delta2 (128 B each) | IC[0..l] (64 B each), Fq-M:
// the vk block zkr_synth_setup emits
extern "C" int zkr_vkey_load_bin(zkr_ctx* ctx, const void* buf, size_t len, zkr_vkey** out) {
    if (!ctx || !buf || !out) {
        set_error("zkr_vkey_load_bin: null argument");
        return ZKR_E_INVALID;
    }
    *out = nullptr;
    if (len < 576 + 64 || (len - 576) % 64) {
        set_error("verification key buffer: length %zu is not 576 + 64 (nPublic + 1)", len);
        return ZKR_E_BADKEY;
    }
    const uint8_t* b = (const uint8_t*)buf;
    VKeyRaw raw;
    raw.n_public = (uint32_t)((len - 576) / 64 - 1);
    memcpy(raw.alfa1, b, 64);
    memcpy(raw.beta2, b + 192, 128);
    memcpy(raw.gamma2, b + 320, 128);
    memcpy(raw.delta2, b + 448, 128);
    raw.ic.assign(b + 576, b + len);
    return vkey_finish(ctx, raw, out);
}

extern "C" void zkr_vkey_free(zkr_vkey* vk) {
    if (!vk) return;
    if (vk->ic_bases) zkr_bases_free(vk->ic_bases);
    delete vk;
}

extern "C" int zkr_vkey_info(const zkr_vkey* vk, uint32_t* n_public) {
    if (!vk) return ZKR_E_INVALID;
    if (n_public) *n_public = vk->n_public;
    return ZKR_OK;
}

extern "C" int zkr_verify(zkr_ctx* ctx, const zkr_vkey* vk, const void* proof, const void* public_signals,
                          size_t n_public, int* valid) {
    if (!ctx || !vk || !proof || !valid || vk->ctx != ctx || (n_public && !public_signals)) {
        set_error("zkr_verify: bad arguments");
        return ZKR_E_INVALID;
    }
    *valid = 0;
    if (n_public != vk->n_public) {      // require(input.length + 1 == vk.IC.length, "verifier-bad-input")  TxVerifier.sol:261
        set_error("verifier-bad-input: %zu public signals given, the key has %u", n_public, vk->n_public);
        return ZKR_E_INVALID;
    }
    const uint8_t* pb = (const uint8_t*)proof;
    pr::G1A a, c;
    pr::G2A b;
    if (!pr::g1_from_std(pb, a) || !pr::g2_from_std(pb + 64, b) || !pr::g1_from_std(pb + 192, c)) return ZKR_OK;
    if (!pr::on_curve(a) || !pr::on_curve(b) || !pr::on_curve(c) || !pr::g2_in_subgroup(b)) return ZKR_OK;
    // vk_x = IC[0] + sum input[i] IC[i+1]: GPU MSM over the resident IC tables (range check input[i] < r inside)
    pr::G1A vkx = vk->ic0;
    if (n_public) {
        uint8_t acc[64];
        ZKR_TRY(zkr_msm(ctx, vk->ic_bases, public_signals, n_public, 0, acc));
        pr::G1A s;
        if (!pr::g1_from_std(acc, s)) {
            set_error("zkr_verify: MSM result out of range");
            return ZKR_E_CUDA;
        }
        vkx = pr::g1_add(vkx, s);
    }
    pr::G1A na = a;
    if (!na.inf) na.y = pr::neg(na.y);       // Pairing.negate(proof.A), TxVerifier.sol:270
    const pr::G1A P[4] = {na, vk->alfa1, vkx, c};
    const pr::G2A Q[4] = {b, vk->beta2, vk->gamma2, vk->delta2};
    bool ok = true;
    const bool one = pr::pairing_product_is_one(P, Q, 4, &ok);
    *valid = (ok && one) ? 1 : 0;
    return ZKR_OK;
}

// prod e(P_i, Q_i) == 1 over n <= 8 pairs of standard-form affine points (64 B / 128 B each, all-zero =
// infinity): the alt_bn128 pairing-check predicate TxVerifier.sol:91-116 hands to precompile 8.  Like the
// precompile it FAILS (ZKR_E_INVALID) on coordinates >= q, points off the curve, or G2 points outside the
// order-r subgroup -- which is also what guarantees the Miller loop never meets a degenerate line.  Host-only.
extern "C" int zkr_pairing_check(const void* g1_points, const void* g2_points, size_t n, int* is_one) {
    if (!is_one || n > 8 || (n && (!g1_points || !g2_points))) {
        set_error("zkr_pairing_check: bad arguments (at most 8 pairs)");
        return ZKR_E_INVALID;
    }
    *is_one = 0;
    pr::G1A P[8];
    pr::G2A Q[8];
    for (size_t i = 0; i < n; i++) {
        if (!pr::g1_from_std((const uint8_t*)g1_points + 64 * i, P[i]) || !pr::g2_from_std((const uint8_t*)g2_points + 128 * i, Q[i]) ||
            !pr::on_curve(P[i]) || !pr::on_curve(Q[i]) || !pr::g2_in_subgroup(Q[i])) {
            set_error("zkr_pairing_check: pair %zu is not a valid (G1, G2) input", i);
            return ZKR_E_INVALID;
        }
    }
    bool ok = true;
    const bool one = pr::pairing_product_is_one(P, Q, (int)n, &ok);
    if (!ok) {
        set_error("zkr_pairing_check: degenerate line (internal)");
        return ZKR_E_INVALID;
    }
    *is_one = one ? 1 : 0;
    return ZKR_OK;
}
