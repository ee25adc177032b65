// Helpers shared by the setup ceremony (ceremony.cu: keys from powers, phase-2 contributions) and phase 1 (powers.cu:
// contributions to the powers of tau and their verification).  Everything here has internal linkage: each file
// that includes it gets its own copy of the kernels and host functions.
#pragma once
#include <algorithm>
#include <cstring>
#include <thread>
#include <vector>

#include "common.cuh"
#include "ec.cuh"
#include "host_ec.cuh"

namespace {
using namespace zkr;

constexpr int kDigits = 64;            // 4-bit signed windows of a scalar < r < 2^254: the top one never carries out
constexpr int kTabLog = 14;            // k_scale_points' tables: tau'^k = lo[k mod 2^14] * hi[k >> 14], k < 2^28
constexpr uint32_t kTab = 1u << kTabLog;

// ------------------------------------------------------------------------------------------------ device

template <class F>
__device__ __forceinline__ void store_key_point(const XYZZ<F>& p, Affine<F>* out) {
    Affine<F> a = {F::zero(), F::one()};      // infinity as binarifyProvingKey writes it: (0, R mod q)
    if (!p.is_inf()) a = p.to_affine();
    a.store(out);
}

__global__ void k_generators(G1Affine* g1, G2Affine* g2) {
    generator<Fq>().store(g1);
    generator<Fq2>().store(g2);
}

// pts[k] = s_k pts[k] in place, key encoding in and out, one thread per point.  s_k = lo[k mod 2^14] hi[k >> 14]
// (Montgomery form; 1 when lo is null) times *c_std (std form; 1 when c_std is null).
// The scalar's signed 4-bit windows d_w in [-7, 8] are the nibbles of s + 0x77..7 minus 7 (s < r < 2^254, so the sum
// does not carry out of 256 bits).  They are read from the top by shifting the sum left, so the digits stay in
// registers; all 64 windows run, as the identity doubles for free.
template <class F>
__global__ void k_scale_points(Affine<F>* pts, size_t n, const Fr* __restrict__ lo, const Fr* __restrict__ hi,
                               const Fr* c_std) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Fr s = lo ? Fr::load_ro(lo + (k & (kTab - 1))) * Fr::load_ro(hi + (k >> kTabLog)) : Fr::one();
    if (c_std) s = s * Fr::load(c_std).to_mont();
    s = s.from_mont();
    uint32_t d[8];
    uint64_t cy = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        cy += (uint64_t)s.v[i] + 0x77777777u;
        d[i] = (uint32_t)cy;
        cy >>= 32;
    }
    const Affine<F> a = Affine<F>::load(pts + k);
    XYZZ<F> acc = XYZZ<F>::identity();
    if (!a.is_inf()) {
        XYZZ<F> t[8];       // t[j - 1] = j a
        t[0] = XYZZ<F>::from_affine(a);
#pragma unroll 1
        for (int j = 1; j < 8; j++) {
            t[j] = t[j - 1];
            t[j].madd(a);
        }
#pragma unroll 1
        for (int w = kDigits - 1; w >= 0; w--) {
#pragma unroll 1
            for (int b = 0; b < 4; b++) acc = acc.dbl();
            const int dg = (int)(d[7] >> 28) - 7;
#pragma unroll
            for (int i = 7; i > 0; i--) d[i] = d[i] << 4 | d[i - 1] >> 28;
            d[0] <<= 4;
            if (dg > 0) acc.add(t[dg - 1]);
            else if (dg < 0) acc.add(t[-dg - 1].neg());
        }
    }
    store_key_point(acc, pts + k);
}

// z[j] = k[j] + c[j] s[j] mod r, std form: the responses of n Schnorr proofs (secret s, nonce k, challenge c)
__global__ void k_schnorr_z(const Fr* s, const Fr* k, const Fr* c, Fr* z, int n) {
    for (int j = 0; j < n; j++) z[j] = (k[j].to_mont() + c[j].to_mont() * s[j].to_mont()).from_mont();
}

// z * P0 == P2 + c * P1 ?   (P0 = P_old, P1 = P_new, P2 = R; zc = z | c std form)
__global__ void k_schnorr_check(const G1Affine* pts, const Fr* zc, int* ok) {
    const G1XYZZ lhs = scalar_mul(G1XYZZ::from_affine(pts[0]), zc[0]);
    G1XYZZ rhs = scalar_mul(G1XYZZ::from_affine(pts[1]), zc[1]);
    rhs.add(G1XYZZ::from_affine(pts[2]));
    if (lhs.is_inf() || rhs.is_inf()) {
        *ok = lhs.is_inf() && rhs.is_inf();
        return;
    }
    const G1Affine a = lhs.to_affine(), b = rhs.to_affine();
    *ok = a.x == b.x && a.y == b.y;
}

// ------------------------------------------------------------------------------------------------ host

void wipe(void* p, size_t n) {
    volatile uint8_t* v = (volatile uint8_t*)p;
    for (size_t i = 0; i < n; i++) v[i] = 0;
}

// Host copy of a call's secrets, wiped when it goes out of scope, on error paths too
template <size_t N>
struct HostSecret {
    uint8_t b[N];
    ~HostSecret() { wipe(b, N); }
};

bool lt_r(const uint8_t* b32) {
    uint32_t v[8];
    memcpy(v, b32, 32);
    for (int i = 7; i >= 0; i--)
        if (v[i] != kRModulus[i]) return v[i] < kRModulus[i];
    return false;
}
bool is_zero32(const uint8_t* b32) {
    uint8_t acc = 0;
    for (int i = 0; i < 32; i++) acc |= b32[i];
    return acc == 0;
}
// a uniform scalar in [1, r) from the OS CSPRNG, 32 B std form
int draw_nonzero(uint8_t* out32) {
    do ZKR_TRY(draw_scalar(out32));
    while (is_zero32(out32));
    return ZKR_OK;
}
// b32 -= r while b32 >= r  (a 256-bit value is below 6 r)
void reduce_r(uint8_t* b32) {
    while (!lt_r(b32)) {
        uint32_t v[8];
        memcpy(v, b32, 32);
        uint64_t borrow = 0;
        for (int i = 0; i < 8; i++) {
            const uint64_t d = (uint64_t)v[i] - kRModulus[i] - borrow;
            v[i] = (uint32_t)d;
            borrow = (d >> 63) & 1;
        }
        memcpy(b32, v, 32);
    }
}

// ---- SHA-256 (FIPS 180-4), host, for the contribution challenge
struct Sha256 {
    uint32_t h[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
    uint8_t buf[64];
    size_t fill = 0;
    uint64_t bits = 0;

    static uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
    void block(const uint8_t* p) {
        static const uint32_t K[64] = {
            0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u,
            0xd807aa98u, 0x12835b01u, 0x243185beu, 0x550c7dc3u, 0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u,
            0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu, 0x2de92c6fu, 0x4a7484aau, 0x5cb0a9dcu, 0x76f988dau,
            0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u, 0x06ca6351u, 0x14292967u,
            0x27b70a85u, 0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u, 0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u,
            0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u, 0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u,
            0x19a4c116u, 0x1e376c08u, 0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu, 0x682e6ff3u,
            0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u, 0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u};
        uint32_t w[64];
        for (int i = 0; i < 16; i++) w[i] = (uint32_t)p[4 * i] << 24 | (uint32_t)p[4 * i + 1] << 16 | (uint32_t)p[4 * i + 2] << 8 | p[4 * i + 3];
        for (int i = 16; i < 64; i++) {
            const uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
            const uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
        for (int i = 0; i < 64; i++) {
            const uint32_t t1 = hh + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
            const uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
            hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    void update(const void* data, size_t n) {
        const uint8_t* p = (const uint8_t*)data;
        bits += 8ull * n;
        while (n) {
            const size_t k = std::min(n, 64 - fill);
            memcpy(buf + fill, p, k);
            fill += k;
            p += k;
            n -= k;
            if (fill == 64) {
                block(buf);
                fill = 0;
            }
        }
    }
    void final(uint8_t out[32]) {
        const uint64_t total = bits;
        const uint8_t pad = 0x80;
        update(&pad, 1);
        const uint8_t zero = 0;
        while (fill != 56) update(&zero, 1);
        uint8_t len[8];
        for (int i = 0; i < 8; i++) len[i] = (uint8_t)(total >> (56 - 8 * i));
        update(len, 8);
        for (int i = 0; i < 8; i++)
            for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(h[i] >> (24 - 8 * j));
    }
};

const char* point_problem(int code) {
    switch (code) {
        case PT_INFINITY: return "is the point at infinity";
        case PT_RANGE: return "has a coordinate >= q";
        case PT_SUBGROUP: return "is not in the order-r subgroup";
        default: return "is not on the curve";
    }
}
// The first of the n points at pts (64 B each for group 1, 128 B for group 2) that fails host_point_check without the
// subgroup test, or n; *code is its PointCheck code.  With inf_y, infinity written as (0, inf_y) passes: the key's
// encoding, inf_y = R mod q.  Threaded.
size_t first_bad_point(int group, const void* pts, size_t n, const void* inf_y, int* code) {
    const size_t sz = group == 1 ? 64 : 128;
    const unsigned nt = std::max(1u, std::min({std::thread::hardware_concurrency(), 16u, (unsigned)(n / 4096) + 1}));
    std::vector<size_t> bad(nt, n);
    std::vector<int> cd(nt, PT_OK);
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++)
        th.emplace_back([&, t] {
            for (size_t i = n * t / nt; i < n * (t + 1) / nt; i++) {
                const uint8_t* pt = (const uint8_t*)pts + sz * i;
                const int c = host_point_check(group, pt, false);
                if (c != PT_OK && !(c == PT_INFINITY && inf_y && !memcmp(pt + sz / 2, inf_y, sz / 2))) {
                    bad[t] = i;
                    cd[t] = c;
                    return;
                }
            }
        });
    for (auto& t : th) t.join();
    for (unsigned t = 0; t < nt; t++)
        if (bad[t] < n) {
            *code = cd[t];
            return bad[t];
        }
    *code = PT_OK;
    return n;
}

// count >= need points given (errors name the entry point fn), and the first `used` of them (every point the setup reads) valid
int check_section(const char* fn, const char* name, int group, const void* pts, uint32_t count, uint32_t need, uint32_t used) {
    if (count < need || !pts) {
        set_error("%s: %s has %u points, %u needed", fn, name, pts ? count : 0u, need);
        return ZKR_E_INVALID;
    }
    int code;
    const size_t bad = first_bad_point(group, pts, used, nullptr, &code);
    if (bad < used) {
        set_error("%s: %s[%zu] %s", fn, name, bad, point_problem(code));
        return ZKR_E_INVALID;
    }
    return ZKR_OK;
}

// gen = the G1 and G2 generators in the key encoding, 64 + 128 B
int generators(zkr_ctx* ctx, cudaStream_t st, uint8_t gen[192]) {
    DevAllocs a;
    G1Affine* d_g1;
    G2Affine* d_g2;
    ZKR_TRY(a.alloc(&d_g1, 64));
    ZKR_TRY(a.alloc(&d_g2, 128));
    ZKR_LAUNCH(ctx, k_generators, 1, 1, 0, st, d_g1, d_g2);
    ZKR_CUDA(cudaMemcpyAsync(gen, d_g1, 64, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaMemcpyAsync(gen + 64, d_g2, 128, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

// c = SHA-256(tag | P_old | P_new | R) as a little-endian integer mod r: the challenge of a Schnorr proof of knowledge
// of s for P_new = s P_old (G1, key encoding)
void challenge(const char* tag, const uint8_t* p_old, const uint8_t* p_new, const uint8_t* R, uint8_t c[32]) {
    Sha256 s;
    s.update(tag, strlen(tag));
    s.update(p_old, 64);
    s.update(p_new, 64);
    s.update(R, 64);
    s.final(c);
    reduce_r(c);
}

// *ok = (z P_old == R + c P_new) for the challenge c of (tag, P_old, P_new, R); points checked, z < r
int schnorr_holds(zkr_ctx* ctx, cudaStream_t st, const char* tag, const uint8_t* p_old, const uint8_t* p_new,
                  const uint8_t* R, const uint8_t* z, bool* ok) {
    uint8_t pts[192], zc[64];
    memcpy(pts, p_old, 64);
    memcpy(pts + 64, p_new, 64);
    memcpy(pts + 128, R, 64);
    memcpy(zc, z, 32);
    challenge(tag, p_old, p_new, R, zc + 32);
    DevAllocs a;
    G1Affine* d_pts;
    Fr* d_zc;
    int* d_ok;
    int flag = 0;
    ZKR_TRY(a.upload(&d_pts, pts, 3, st));
    ZKR_TRY(a.upload(&d_zc, zc, 2, st));
    ZKR_TRY(a.alloc(&d_ok, sizeof(int)));
    ZKR_LAUNCH(ctx, k_schnorr_check, 1, 1, 0, st, d_pts, d_zc, d_ok);
    ZKR_CUDA(cudaMemcpyAsync(&flag, d_ok, sizeof(int), cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    *ok = flag != 0;
    return ZKR_OK;
}

}  // namespace
