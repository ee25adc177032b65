// Radix-2^k NTT over BN254 Fr and the H = (A.B - C)/Z pipeline.
//
// Replaces websnark fft_ifft / fft_fft / fft_mulN inside calcH of groth16GenProof
// (/root/reference/operator/src/snarks/common.ts:29) and snarkjs PolField.ifft / mul
// (prover_groth.js calculateH).  omega_k = 5^((r-1)/2^k) as in snarkjs polfield.js.
//
// Structure (DESIGN.md "NTT"):
//   * N = 2^n is split into <= 3 passes of <= 11 bits (four-step / Bailey).  One pass = one kernel:
//     a CTA stages a tile of 2^k rows x 2^c adjacent columns (<= 2048 elements, 72 KB) in shared
//     memory with coalesced 128-bit loads, runs the 2^k-point sub-NTT in radix-8 register stages
//     (each thread owns 8 elements = 3 butterfly levels between two __syncthreads), applies the
//     inter-pass twiddle omega_N'^(col * rev(row)) in registers, and streams the tile back.
//   * shared memory is limb-major (8 planes of u32) with a 1-in-8 pad so every register-stage
//     access pattern is bank-conflict free (or 2-way at worst).
//   * DIF (natural in, bit-reversed out) and its transpose DIT (bit-reversed in, natural out) share
//     the kernel; the prover chains DIF^-1 -> DIT -> DIF^-1 so no bit-reversal pass is ever run.
//   * data may be in standard OR Montgomery form: every constant (twiddles, scalings) is stored in
//     Montgomery form and mont_mul(x, cR) = x*c keeps the form of x.
#include <cstdlib>
#include <cstring>

#include "ntt_iface.cuh"

namespace zkr {

constexpr int kTileLog = 11;

namespace {

__device__ __forceinline__ Fr fr_const(const uint32_t (&l)[8]) {
    Fr r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = l[i];
    return r;
}

__device__ __forceinline__ Fr fr_pow(Fr base, unsigned long long e) {
    Fr acc = Fr::one();
    while (e) {
        if (e & 1) acc = acc * base;
        base = base.sqr();
        e >>= 1;
    }
    return acc;
}

__global__ void k_ntt_roots(NttRoots* out, int log_n) {
    // omega_28 = 5^((r-1)/2^28), Montgomery form (KAT: SURVEY.md B.1)
    const uint32_t W28[8] = {0x80d13d9cu, 0x636e7355u, 0x2445ffd6u, 0xa22bf374u,
                             0x1eb203d8u, 0x56452ac0u, 0x2963f9e7u, 0x1860ef94u};
    const uint32_t INV2[8] = {0x1ffffffeu, 0x783c14d8u, 0x0c8d1eddu, 0xaf982f6fu,
                              0xfcfd4f45u, 0x8f5f7492u, 0x3d9cbfacu, 0x1f37631au};
    Fr g = fr_const(W28);
    for (int i = 28; i > log_n + 1; i--) g = g.sqr();
    Fr w = g.sqr();
    Fr nn = Fr::zero();
    nn.v[0] = 1u << log_n;
    nn = nn.to_mont();
    NttRoots r;
    r.w = w;
    r.wi = w.inverse();
    r.g = g;
    r.gi = g.inverse();
    r.ninv = nn.inverse();
    r.hconst = Fr::r2() * r.ninv * fr_const(INV2);   // Montgomery form of R/(2N)
    r.one = Fr::one();
    *out = r;
}

// out[i] = cst * base^(i * stride)
__global__ void k_pow_table(Fr* out, unsigned count, const Fr* base, unsigned long long stride, const Fr* cst) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Fr v = fr_pow(*base, (unsigned long long)i * stride);
    if (cst) v = v * *cst;
    v.store(out + i);
}

// out[(row << s) + col] = omega^((col * rev_k(row)) << tw_shift): the inter-pass twiddles of one pass, in the layout of a chunk
__global__ void k_twfull(Fr* out, int chunk_log, int k, int tw_shift, const Fr* lo, const Fr* hi, int lb) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >> chunk_log) return;
    const int s = chunk_log - k;
    const unsigned row = (unsigned)(idx >> s), col = (unsigned)(idx & (((size_t)1 << s) - 1));
    const unsigned rev = __brev(row) >> (32 - k);
    const unsigned X = (col * rev) << tw_shift;
    (Fr::load_ro(lo + (X & ((1u << lb) - 1))) * Fr::load_ro(hi + (X >> lb))).store(out + idx);
}

// out[p] = lo[j & mask] * hi[j >> lb] at j = bitrev(p): a two-level power table spread out in bit-reversed order
__global__ void k_pow_bitrev(Fr* out, int log_n, const Fr* lo, const Fr* hi, int lb) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >> log_n) return;
    const unsigned j = __brev((unsigned)p) >> (32 - log_n);
    (Fr::load_ro(lo + (j & ((1u << lb) - 1))) * Fr::load_ro(hi + (j >> lb))).store(out + p);
}

// out[p] = c * g^j(p), standard form; c, g standard form.  j(p) = start + p (world_log < 0) or the transform index of
// local element p of rank's COLS slab (see k_scale_pow_sharded, layout 0).  Workload generator: a dense vector whose
// transform has a closed form on the host, X[k] = c (g^N - 1) / (g w^k - 1)  (bench.py, tests).
__global__ void k_fill_geometric(Fr* out, size_t n_local, const Fr* cg, unsigned long long start, int s0, int world_log,
                                 int rank) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_local) return;
    unsigned long long j;
    if (world_log < 0) {
        j = start + p;
    } else {
        const int cl = s0 - world_log;
        j = ((p >> cl) << s0) + ((unsigned long long)rank << cl) + (p & (((size_t)1 << cl) - 1));
    }
    const Fr c = Fr::load(cg), g = Fr::load(cg + 1).to_mont();
    (c * fr_pow(g, j)).store(out + p);
}

__device__ __forceinline__ int slot_of(int e) { return e + (e >> 3); }

// MODE selects where the tile is written back (the multi-GPU four-step exchange is fused into the pass):
//   0  in place (single GPU, and the local passes of a sharded transform)
//   1  COLS slab in, push to the peers' ROWS buffers: row i of the first DIF pass belongs to rank i >> (k - g)
//   2  push to the peers' COLS buffers: column j of the last-but-one DIT pass belongs to rank j >> (s0 - g)
//   3  in place on a COLS slab (last DIT pass)
// On a COLS slab (modes 1, 3) ls_ = log2 of the row stride in memory (s0 - g) and ctw_ = global column of
// this rank's first local column (twiddles use global coordinates); otherwise ls == s and ctw == 0.
// Fused element-wise work (H pipeline: no separate sweeps over memory).  Runtime values, uniform per launch:
//   ld_op  LD_PLAIN | LD_MUL2: element = src[pos] * in2[pos] (S = A_T.B_T and P = A.B are formed while the first pass of
//          their transform loads its tile) | LD_TAB: element = data[pos] * tab[pos] (coset scaling g^j / N, table stored
//          in the order of the data)
//   st_op  ST_PLAIN | ST_HFINAL: out[pos] = in2[pos] * K - x * tab[pos]   (h = S K - P g^-j K, see h_pipeline)
// twfull != null: the inter-pass twiddle omega_N'^(col * rev(row)) comes from ONE table laid out like a chunk of the
// data (coalesced like the data itself, one modmul per element) instead of the product of two sqrt(N)-sized tables
// (two modmuls per element).  pos = position in the whole vector (MODE 0 only).
enum { LD_PLAIN = 0, LD_MUL2 = 1, LD_TAB = 2 };
enum { ST_PLAIN = 0, ST_HFINAL = 1 };
struct PassFuse {
    const Fr* src;       // LD_MUL2: first operand (null = data)
    const Fr* in2;       // LD_MUL2: second operand; ST_HFINAL: S
    const Fr* tab;       // LD_TAB / ST_HFINAL: table indexed by position
    const Fr* kconst;    // ST_HFINAL: K
    Fr* out;             // ST_HFINAL: destination (null = data)
    const Fr* twfull;    // full inter-pass twiddle table of this pass (null = two-level)
    Fr* data2;           // second vector transformed by the same launch (blockIdx.y == 1); null = one vector
    int ld_op, st_op;
};

// RL = log2 of the register-stage radix.  RL = 3 (the only instantiation): a thread holds 8 elements = 3 butterfly levels
// between two barriers, 112-128 registers, 2 CTAs / SM (4 warps per scheduler).  RL = 2 (two groups of 4 elements,
// 2 levels per barrier, 80 registers, 3 CTAs / SM) was built and timed in round 2: 1-12 % SLOWER at every size
// (profiles/r02_ntt_radix_ab.json) -- the extra shared-memory round trip per pass costs more than the extra warps hide.
template <bool DIT, int MODE, int RL>
__global__ void __launch_bounds__(256, RL == 3 ? 2 : 3)
k_ntt_pass(Fr* data, int k, int c, int s, int ls_, int chunk_log, unsigned ctw_, const Fr* __restrict__ W,
           int kw, const Fr* __restrict__ tlo, const Fr* __restrict__ thi, int lb, int tw_shift, NttXchg xp, PassFuse fz) {
    extern __shared__ uint32_t sm[];
    constexpr bool kSlab = MODE == 1 || MODE == 3;
    const int ls = kSlab ? ls_ : s;
    const unsigned ctw = kSlab ? ctw_ : 0u;
    const int T = k + c;
    const int tile = 1 << T;
    const int plane = tile + (tile >> 3) + 4;
    const int tid = threadIdx.x;
    const unsigned cgmask = (1u << (ls - c)) - 1;
    const unsigned cg = blockIdx.x & cgmask;
    const size_t q = blockIdx.x >> (ls - c);
    // two independent transforms of one size can share a launch (the H pipeline's A and B): twice the CTAs per wave
    // quantum, half the launches
    if (MODE == 0 && blockIdx.y) data = fz.data2;
    Fr* chunk = data + (q << chunk_log);
    const unsigned cm = cg << c;             // first column of the tile in memory
    const unsigned c0 = ctw + cm;            // ... and in the transform's global coordinates
    const int cmask = (1 << c) - 1;

    const unsigned lbmask = (1u << lb) - 1;
    // ---- global -> shared.  blockDim.x == tile / 8 (launch_pass), so every thread moves exactly 8 elements = 16
    // 16-byte units; the loads of a group are all issued before the first shared store (an un-unrolled loop exposed
    // one HBM latency per unit: 12 % of the pass in the round-1 ncu source view, profiles/r01_ncu_ntt_pass.md).
    const size_t qbase = q << chunk_log;      // position of the chunk in the whole vector (fused ops, MODE 0)
    if ((DIT && s > 0) || fz.ld_op != LD_PLAIN) {
        // Whole elements per thread.  DIT applies the inter-pass twiddle omega_N'^(col * rev(row)) BEFORE its butterflies:
        // do it on the way in, so the register stages below hold nothing but the 8 butterfly operands (with the twiddle
        // inside the first stage ptxas spilled 272 B per thread).  The fused load operations ride on the same path.
        const Fr* src = fz.src ? fz.src + qbase : chunk;
#pragma unroll 1
        for (int g = 0; g < 2; g++) {
            Fr v[4];
            size_t off[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int e = tid + (g * 4 + i) * (tile >> 3);
                off[i] = ((size_t)(e >> c) << ls) + cm + (e & cmask);
                v[i] = Fr::load(src + off[i]);
            }
            if (fz.ld_op == LD_MUL2) {
#pragma unroll
                for (int i = 0; i < 4; i++) v[i] = v[i] * Fr::load(fz.in2 + qbase + off[i]);
            } else if (fz.ld_op == LD_TAB) {
#pragma unroll
                for (int i = 0; i < 4; i++) v[i] = v[i] * Fr::load_ro(fz.tab + qbase + off[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int e = tid + (g * 4 + i) * (tile >> 3);
                if (DIT && s > 0) {
                    if (fz.twfull) {
                        v[i] = v[i] * Fr::load_ro(fz.twfull + ((size_t)(e >> c) << s) + c0 + (e & cmask));
                    } else {
                        const unsigned rev = __brev((unsigned)(e >> c)) >> (32 - k);
                        const unsigned X = ((c0 + (e & cmask)) * rev) << tw_shift;
                        v[i] = v[i] * (Fr::load_ro(tlo + (X & lbmask)) * Fr::load_ro(thi + (X >> lb)));
                    }
                }
                uint32_t* d = sm + slot_of(e);
#pragma unroll
                for (int l = 0; l < 8; l++) d[l * plane] = v[i].v[l];
            }
        }
    } else {
#pragma unroll 1
        for (int g = 0; g < 2; g++) {
            uint4 v[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int u = tid + (g * 8 + i) * (tile >> 3);
                const int e = u >> 1;
                v[i] = *(reinterpret_cast<const uint4*>(chunk + ((size_t)(e >> c) << ls) + cm + (e & cmask)) + (u & 1));
            }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int u = tid + (g * 8 + i) * (tile >> 3);
                uint32_t* d = sm + (4 * (u & 1)) * plane + slot_of(u >> 1);
                d[0] = v[i].x;
                d[plane] = v[i].y;
                d[2 * plane] = v[i].z;
                d[3 * plane] = v[i].w;
            }
        }
    }
    __syncthreads();

    constexpr int G = 1 << RL;                // elements per register group
    int bit = DIT ? c : T - 1;
    while (DIT ? (bit <= T - 1) : (bit >= c)) {
        int lo, act_lo, act_hi;
        if (DIT) {
            lo = bit > T - RL ? T - RL : bit;
            act_lo = bit;
            act_hi = lo + RL - 1;
        } else {
            lo = bit < RL - 1 ? 0 : bit - (RL - 1);
            act_hi = bit;
            act_lo = lo > c ? lo : c;
        }
        const bool tw_now = !DIT && (s > 0) && (act_lo == c);     // DIF: after the last butterfly level (DIT: at load)
#pragma unroll 1
        for (int grp = 0; grp < (8 >> RL); grp++) {
            const int gid = tid + grp * (tile >> 3);
            const int base = ((gid >> lo) << (lo + RL)) | (gid & ((1 << lo) - 1));
            Fr x[G];
#pragma unroll
            for (int j = 0; j < G; j++) {
                const uint32_t* p = sm + slot_of(base + (j << lo));
#pragma unroll
                for (int l = 0; l < 8; l++) x[j].v[l] = p[l * plane];
            }
#pragma unroll
            for (int ii = 0; ii < RL; ii++) {
                const int i = DIT ? ii : RL - 1 - ii;
                const int p = lo + i;
                if (p < act_lo || p > act_hi) continue;
                const int pc = p - c;                  // butterfly half-size = 2^pc rows
#pragma unroll
                for (int jl = 0; jl < (1 << i); jl++) {
                    Fr w;
                    if (pc > 0) {
                        unsigned rowbits = ((unsigned)(base | (jl << lo)) >> c) & ((1u << pc) - 1);
                        w = Fr::load_ro(W + ((size_t)rowbits << (kw - 1 - pc)));
                    }
#pragma unroll
                    for (int ju = 0; ju < (1 << (RL - 1 - i)); ju++) {
                        const int j0 = jl | (ju << (i + 1));
                        const int j1 = j0 | (1 << i);
                        if (DIT) {
                            if (pc > 0) x[j1] = x[j1] * w;
                            const Fr u = x[j0], v = x[j1];
                            x[j0] = u + v;
                            x[j1] = u - v;
                        } else {
                            Fr u = x[j0], v = x[j1];
                            x[j0] = u + v;
                            Fr d = u - v;
                            x[j1] = pc > 0 ? d * w : d;
                        }
                    }
                }
            }
            if (!DIT && tw_now) {
                if (fz.twfull) {
                    // software-pipelined: the table entry of element j + 1 is in flight while element j is multiplied
                    // (r02 ncu: 14 % of the pass's stall samples were long_sb on the first IMAD.WIDE behind each load)
                    auto tw_at = [&](int j) {
                        const int e = base + (j << lo);
                        return Fr::load_ro(fz.twfull + ((size_t)(e >> c) << s) + c0 + (e & cmask));
                    };
                    Fr tnext = tw_at(0);
#pragma unroll
                    for (int j = 0; j < G; j++) {
                        const Fr t = tnext;
                        if (j + 1 < G) tnext = tw_at(j + 1);
                        x[j] = x[j] * t;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < G; j++) {
                        int e = base + (j << lo);
                        unsigned rho = e >> c, col = e & cmask;
                        unsigned rev = __brev(rho) >> (32 - k);
                        unsigned X = ((c0 + col) * rev) << tw_shift;
                        x[j] = x[j] * (Fr::load_ro(tlo + (X & lbmask)) * Fr::load_ro(thi + (X >> lb)));
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < G; j++) {
                uint32_t* p = sm + slot_of(base + (j << lo));
#pragma unroll
                for (int l = 0; l < 8; l++) p[l * plane] = x[j].v[l];
            }
        }
        __syncthreads();
        bit = DIT ? act_hi + 1 : act_lo - 1;
    }

    // ---- shared -> global
    if (MODE == 0 && fz.st_op == ST_HFINAL) {
        // whole elements: out[pos] = S[pos] * K - x * tab[pos]
        const Fr K = Fr::load_ro(fz.kconst);
        Fr* outp = (fz.out ? fz.out : data) + qbase;
#pragma unroll 2
        for (int e = tid; e < tile; e += blockDim.x) {
            const size_t off = ((size_t)(e >> c) << ls) + cm + (e & cmask);
            Fr x;
            const uint32_t* d = sm + slot_of(e);
#pragma unroll
            for (int l = 0; l < 8; l++) x.v[l] = d[l * plane];
            const Fr v = Fr::load(fz.in2 + qbase + off) * K - x * Fr::load_ro(fz.tab + qbase + off);
            v.store(outp + off);
        }
        return;
    }
    for (int u = tid; u < 2 * tile; u += blockDim.x) {
        int e = u >> 1, half = u & 1;
        int row = e >> c, col = e & cmask;
        const uint32_t* d = sm + (4 * half) * plane + slot_of(e);
        uint4 v = make_uint4(d[0], d[plane], d[2 * plane], d[3 * plane]);
        Fr* dp;
        if (MODE == 0 || MODE == 3) {
            dp = chunk + ((size_t)row << ls) + cm + col;
        } else if (MODE == 1) {
            const int rl = k - xp.g;         // log2 rows per rank
            dp = xp.peer[row >> rl] + ((size_t)(row & ((1 << rl) - 1)) << xp.s0) + c0 + col;
        } else {
            const unsigned j = ((unsigned)row << s) + cm + col;                 // column inside row-chunk q
            const int cl = xp.s0 - xp.g;     // log2 columns per rank
            const size_t i = ((size_t)xp.rank << (xp.k0 - xp.g)) + q;           // global row
            dp = xp.peer[j >> cl] + (i << cl) + (j & ((1u << cl) - 1));
        }
        *(reinterpret_cast<uint4*>(dp) + half) = v;
    }
}

// N = 2 or 4: one thread, direct DFT
__global__ void k_ntt_tiny(Fr* data, int log_n, const Fr* root, bool bitrev_in, bool bitrev_out) {
    int n = 1 << log_n;
    Fr x[4], y[4];
    for (int i = 0; i < n; i++) {
        int pos = bitrev_in ? (int)(__brev(i) >> (32 - log_n)) : i;
        x[i] = Fr::load(data + pos);
    }
    Fr w = *root;
    for (int kk = 0; kk < n; kk++) {
        Fr acc = Fr::zero();
        Fr wk = fr_pow(w, kk), t = Fr::one();
        for (int i = 0; i < n; i++) {
            acc = acc + x[i] * t;
            t = t * wk;
        }
        y[kk] = acc;
    }
    for (int kk = 0; kk < n; kk++) {
        int pos = bitrev_out ? (int)(__brev(kk) >> (32 - log_n)) : kk;
        y[kk].store(data + pos);
    }
}

__global__ void k_pointwise_mul(Fr* out, const Fr* a, const Fr* b, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    (Fr::load(a + i) * Fr::load(b + i)).store(out + i);
}

// x[p] *= lo[j & mask] * hi[j >> lb],  j = bitrev(p) or p
__global__ void k_scale_pow(Fr* x, size_t n, int log_n, const Fr* lo, const Fr* hi, int lb, bool bitrev_idx) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    unsigned j = bitrev_idx ? (__brev((unsigned)p) >> (32 - log_n)) : (unsigned)p;
    Fr t = Fr::load_ro(lo + (j & ((1u << lb) - 1))) * Fr::load_ro(hi + (j >> lb));
    (Fr::load(x + p) * t).store(x + p);
}

// sharded variant: j = transform index of local element p of a COLS (natural) or ROWS (bit-reversed) slab
__global__ void k_scale_pow_sharded(Fr* x, size_t n_local, int log_n, const Fr* lo, const Fr* hi, int lb, int layout,
                                    int s0, int g, int rank) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_local) return;
    unsigned j;
    if (layout == 0) {
        const int cl = s0 - g;
        j = (unsigned)(((p >> cl) << s0) + ((size_t)rank << cl) + (p & (((size_t)1 << cl) - 1)));
    } else {
        const unsigned pos = (unsigned)(((size_t)rank << (log_n - g)) + p);
        j = __brev(pos) >> (32 - log_n);
    }
    Fr t = Fr::load_ro(lo + (j & ((1u << lb) - 1))) * Fr::load_ro(hi + (j >> lb));
    (Fr::load(x + p) * t).store(x + p);
}

__global__ void k_scale_const(Fr* x, size_t n, const Fr* cst) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    (Fr::load(x + p) * *cst).store(x + p);
}

// out[bitrev(p)] = x[p] * cst * (lo/hi power of j = bitrev(p), if lo != null)
__global__ void k_bitrev_scale(Fr* out, const Fr* x, size_t n, int log_n, const Fr* cst, const Fr* lo,
                               const Fr* hi, int lb) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    unsigned j = __brev((unsigned)p) >> (32 - log_n);
    Fr v = Fr::load(x + p);
    if (lo) v = v * (Fr::load_ro(lo + (j & ((1u << lb) - 1))) * Fr::load_ro(hi + (j >> lb)));
    else if (cst) v = v * *cst;
    v.store(out + j);
}

// h[p or bitrev(p)] = S[p] * K - P[p] * (gi^j * K),  j = bitrev(p), K = R/(2N)  (see h_pipeline)
__global__ void k_h_final(Fr* h, const Fr* S, const Fr* P, size_t n, int log_n, const Fr* kconst,
                          const Fr* lo, const Fr* hi, int lb, bool bitrev_out) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    unsigned j = __brev((unsigned)p) >> (32 - log_n);
    Fr t = Fr::load_ro(lo + (j & ((1u << lb) - 1))) * Fr::load_ro(hi + (j >> lb));
    Fr v = Fr::load(S + p) * *kconst - Fr::load(P + p) * t;
    v.store(h + (bitrev_out ? p : (size_t)j));
}

// ZKR_NTT_SPLIT="a[,b[,c[,d]]]" (experiment knob): explicit widths of up to four passes, 3..11 bits each, for the
// transforms whose size they sum to.  Read once per process, like the other NTT knobs: a size's full twiddle tables are
// cached per pass index (get_twfull), so a split that changed between two transforms of one size would pair pass i with
// a table built for another chunk width.
struct SplitKnob {
    int v[4];
    int cnt, sum;
};

const SplitKnob& split_knob() {
    static const SplitKnob knob = [] {
        SplitKnob s = {};
        const char* e = getenv("ZKR_NTT_SPLIT");
        for (const char* q = e; q && *q && s.cnt < 4;) {
            s.v[s.cnt] = atoi(q);
            s.sum += s.v[s.cnt++];
            q = strchr(q, ',');
            if (q) q++;
        }
        for (int i = 0; i < s.cnt; i++)
            if (s.v[i] < 3 || s.v[i] > kTileLog) s.cnt = 0;
        return s;
    }();
    return knob;
}

int plan_passes(int n, int* ks) {
    int np = (n + kTileLog - 1) / kTileLog;
    if (np < 1) np = 1;
    int base = n / np, rem = n % np;
    for (int i = 0; i < np; i++) ks[i] = base + (i < rem ? 1 : 0);
    const SplitKnob& sk = split_knob();
    if (sk.cnt >= 1 && sk.sum == n) {
        for (int i = 0; i < sk.cnt; i++) ks[i] = sk.v[i];
        np = sk.cnt;
    }
    return np;
}

}  // namespace

void ntt_tables_free(NttTables* t) {
    if (!t) return;
    Fr** ps[] = {&t->wsub_f, &t->wsub_i, &t->tw_lo_f, &t->tw_hi_f, &t->tw_lo_i, &t->tw_hi_i, &t->cs_lo,
                 &t->cs_hi, &t->cs_hi_n, &t->ci_lo, &t->ci_hi_n, &t->ci_hi_h};
    for (Fr** p : ps) cudaFree(*p);
    for (int i = 0; i < 4; i++) {
        cudaFree(t->twfull_f[i]);
        cudaFree(t->twfull_i[i]);
    }
    cudaFree(t->cs_br);
    cudaFree(t->hf_br);
    cudaFree(t->roots);
    delete t;
}

static int pow_table(zkr_ctx* ctx, cudaStream_t st, Fr** out, unsigned count, const Fr* base,
                     unsigned long long stride, const Fr* cst, size_t* bytes) {
    ZKR_CUDA(cudaMalloc(out, (size_t)count * sizeof(Fr)));
    *bytes += (size_t)count * sizeof(Fr);
    ZKR_LAUNCH(ctx, k_pow_table, ceil_div(count, 128), 128, 0, st, *out, count, base, stride, cst);
    return ZKR_OK;
}

int ntt_get_tables(zkr_ctx* ctx, int log_n, NttTables** out) {
    auto it = ctx->ntt.find(log_n);
    if (it != ctx->ntt.end()) {
        *out = it->second;
        return ZKR_OK;
    }
    if (log_n < 1 || log_n > 27) {
        set_error("NTT size 2^%d unsupported (1..27)", log_n);
        return ZKR_E_UNSUPPORTED;
    }
    // Function attributes are per device: set them whenever tables are built for a context (cold path, idempotent).
    // A process-wide "done" flag left the > 48 KB opt-in missing on every device but the first one a process used
    // (one process driving several GPUs: zkr_prove_batch / ProofQueue).
    {
#define ZKR_NTT_ATTR(...)                                                                                              \
    ZKR_CUDA(cudaFuncSetAttribute((k_ntt_pass<__VA_ARGS__>), cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); \
    ZKR_CUDA(cudaFuncSetAttribute((k_ntt_pass<__VA_ARGS__>), cudaFuncAttributePreferredSharedMemoryCarveout, 100))
        ZKR_NTT_ATTR(false, 0, 3);
        ZKR_NTT_ATTR(true, 0, 3);
        ZKR_NTT_ATTR(false, 1, 3);
        ZKR_NTT_ATTR(true, 2, 3);
        ZKR_NTT_ATTR(true, 3, 3);
#undef ZKR_NTT_ATTR
    }
    NttTables* t = new NttTables();
    t->log_n = log_n;
    t->kw = log_n < kTileLog ? log_n : kTileLog;
    t->lb = (log_n + 1) / 2;
    cudaStream_t st = ctx->s[0];
    ZKR_CUDA(cudaMalloc(&t->roots, sizeof(NttRoots)));
    ZKR_LAUNCH(ctx, k_ntt_roots, 1, 1, 0, st, t->roots, log_n);
    const unsigned nlo = 1u << t->lb, nhi = 1u << (log_n - t->lb);
    const unsigned long long hs = 1ull << t->lb;
    NttRoots* r = t->roots;
    const unsigned nsub = 1u << (t->kw - 1);
    const unsigned long long sub_stride = 1ull << (log_n - t->kw);
    ZKR_TRY(pow_table(ctx, st, &t->wsub_f, nsub, &r->w, sub_stride, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->wsub_i, nsub, &r->wi, sub_stride, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->tw_lo_f, nlo, &r->w, 1, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->tw_hi_f, nhi, &r->w, hs, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->tw_lo_i, nlo, &r->wi, 1, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->tw_hi_i, nhi, &r->wi, hs, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->cs_lo, nlo, &r->g, 1, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->cs_hi, nhi, &r->g, hs, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->cs_hi_n, nhi, &r->g, hs, &r->ninv, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->ci_lo, nlo, &r->gi, 1, nullptr, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->ci_hi_n, nhi, &r->gi, hs, &r->ninv, &t->bytes));
    ZKR_TRY(pow_table(ctx, st, &t->ci_hi_h, nhi, &r->gi, hs, &r->hconst, &t->bytes));
    ZKR_CUDA(cudaStreamSynchronize(st));
    ctx->ntt[log_n] = t;
    *out = t;
    return ZKR_OK;
}

// one pass = one launch
struct PassGeom {
    int k, c, s, ls, chunk_log, tw_shift;
    unsigned ctw, blocks;
};

template <int MODE>
static int launch_pass(zkr_ctx* ctx, cudaStream_t st, const NttTables* t, Fr* data, const PassGeom& g, bool dit,
                       bool inverse, const NttXchg& xp, double prof_units, const PassFuse& fz = PassFuse{}) {
    const Fr* W = inverse ? t->wsub_i : t->wsub_f;
    const Fr* tlo = inverse ? t->tw_lo_i : t->tw_lo_f;
    const Fr* thi = inverse ? t->tw_hi_i : t->tw_hi_f;
    const int tile = 1 << (g.k + g.c);
    const int threads = tile / 8;
    const size_t smem = (size_t)8 * (tile + (tile >> 3) + 4) * sizeof(uint32_t);
    // the pass whose write-back is the all-to-all (remote stores) is timed on its own: bench.py's exchange GB/s
    const int pid = (MODE == 1 || MODE == 2) ? PROF_NTT_XCHG : PROF_NTT_PASS;
    const dim3 grid(g.blocks, (MODE == 0 && fz.data2) ? 2 : 1);
    const int pslot = ctx->prof_begin(pid, st, prof_units * grid.y);
    if (dit) {
        ZKR_LAUNCH(ctx, (k_ntt_pass<true, MODE == 1 ? 3 : MODE, 3>), grid, threads, smem, st, data, g.k, g.c, g.s,
                   g.ls, g.chunk_log, g.ctw, W, t->kw, tlo, thi, t->lb, g.tw_shift, xp, fz);
    } else {
        ZKR_LAUNCH(ctx, (k_ntt_pass<false, (MODE == 2 || MODE == 3) ? 0 : MODE, 3>), grid, threads, smem, st, data, g.k, g.c, g.s,
                   g.ls, g.chunk_log, g.ctw, W, t->kw, tlo, thi, t->lb, g.tw_shift, xp, fz);
    }
    ctx->prof_end(pid, pslot, st);
    return ZKR_OK;
}

// Full inter-pass twiddle tables are used up to this size (2 x N x 32 B per direction and pass boundary: 1 GB per
// direction at 2^24); above it, and on the sharded paths, the two-level lookup stays.  ZKR_NTT_TWFULL_MAXLOG overrides
// (0 = never: A/B against the round-1 kernel).
static int twfull_maxlog() {
    static const int v = getenv("ZKR_NTT_TWFULL_MAXLOG") ? atoi(getenv("ZKR_NTT_TWFULL_MAXLOG")) : 24;
    return v;
}

// table of pass i (chunk_log, k) for one direction, built on first use (cold path; synchronises the stream once)
static int get_twfull(zkr_ctx* ctx, cudaStream_t st, NttTables* t, int i, int chunk_log, int k, bool inverse, const Fr** out) {
    Fr** slot = inverse ? &t->twfull_i[i] : &t->twfull_f[i];
    if (!*slot) {
        const size_t cnt = (size_t)1 << chunk_log;
        ZKR_CUDA(cudaMalloc(slot, cnt * sizeof(Fr)));
        t->bytes += cnt * sizeof(Fr);
        ZKR_LAUNCH(ctx, k_twfull, ceil_div(cnt, 256), 256, 0, st, *slot, chunk_log, k, t->log_n - chunk_log,
                   inverse ? t->tw_lo_i : t->tw_lo_f, inverse ? t->tw_hi_i : t->tw_hi_f, t->lb);
    }
    *out = *slot;
    return ZKR_OK;
}

// In-place transform of 2^log_n elements on `st`.
//   dit == false: natural in  -> bit-reversed out (DIF)
//   dit == true : bit-reversed in -> natural out  (DIT)
// inverse selects omega^-1; no 1/N scaling is applied here.
// first / last (nullable): fused element-wise work of the first executed pass's load (ld_op, src, in2, tab) and of the
// last executed pass's store (st_op, in2, tab, kconst, out).
static int ntt_run_ex(zkr_ctx* ctx, cudaStream_t st, Fr* data, int log_n, bool dit, bool inverse, const PassFuse* first,
                      const PassFuse* last, Fr* data2 = nullptr) {
    NttTables* t;
    ZKR_TRY(ntt_get_tables(ctx, log_n, &t));
    if (log_n < 3) {
        if (first || last) return ZKR_E_UNSUPPORTED;
        ZKR_LAUNCH(ctx, k_ntt_tiny, 1, 1, 0, st, data, log_n, inverse ? &t->roots->wi : &t->roots->w, dit, !dit);
        return ZKR_OK;
    }
    int ks[4];
    const int np = plan_passes(log_n, ks);
    const NttXchg none = {};
    static const unsigned min_blocks = getenv("ZKR_NTT_MIN_BLOCKS") ? (unsigned)atoi(getenv("ZKR_NTT_MIN_BLOCKS")) : 1024u;   // experiment knob; 0 = full-width tiles always
    for (int step = 0; step < np; step++) {
        const int i = dit ? np - 1 - step : step;
        PassGeom g;
        g.chunk_log = log_n;
        for (int j = 0; j < i; j++) g.chunk_log -= ks[j];
        g.k = ks[i];
        g.s = g.chunk_log - g.k;
        g.c = kTileLog - g.k;
        if (g.c > g.s) g.c = g.s;
        // Transforms of <= 2^20 elements make fewer full-width tiles than the machine has CTA slots (2^17: 64 tiles for
        // 148 SMs; 2^20: 512 tiles for 296 slots = 1.73 waves): narrower tiles spread the same threads over all SMs.
        // The pass is IMAD-bound with DRAM at 2-4 % of peak, so the shorter contiguous segments cost nothing.
        while (g.c > 0 && (1u << (log_n - g.k - g.c)) < min_blocks) g.c--;
        g.ls = g.s;
        g.ctw = 0;
        g.tw_shift = log_n - g.chunk_log;
        g.blocks = 1u << (log_n - g.k - g.c);
        PassFuse fz = {};
        fz.data2 = data2;
        if (first && step == 0) {
            fz.ld_op = first->ld_op;
            fz.src = first->src;
            fz.in2 = first->in2;
            fz.tab = first->tab;
        }
        if (last && step == np - 1) {
            fz.st_op = last->st_op;
            fz.in2 = last->in2;         // a single-pass transform never combines LD_MUL2 with ST_HFINAL's in2: see h_pipeline
            fz.tab = last->tab;
            fz.kconst = last->kconst;
            fz.out = last->out;
        }
        if (g.s > 0 && log_n <= twfull_maxlog()) ZKR_TRY(get_twfull(ctx, st, t, i, g.chunk_log, g.k, inverse, &fz.twfull));
        ZKR_TRY(launch_pass<0>(ctx, st, t, data, g, dit, inverse, none, (double)((size_t)1 << log_n), fz));
    }
    return ZKR_OK;
}

int ntt_run(zkr_ctx* ctx, cudaStream_t st, Fr* data, int log_n, bool dit, bool inverse) {
    return ntt_run_ex(ctx, st, data, log_n, dit, inverse, nullptr, nullptr);
}

// Rows of the sharded four-step, 2^k0.  The passes after the exchange work on contiguous rows of 2^s0
// elements and want full 2^11 tiles, so s0 is 11 (one local pass) up to 2^22 and >= 14 (a short pass + a
// full one) above; k0 <= 9 there keeps >= 4 adjacent columns (128 contiguous bytes) per remote store
// segment.  k0 >= g so that every rank owns whole rows.  ZKR_NTT_SHARD_K0 overrides (experiments).
int ntt_sharded_k0(int log_n, int g) {
    if (const char* e = getenv("ZKR_NTT_SHARD_K0")) {
        const int v = atoi(e);
        if (v >= g && v >= 3 && v <= kTileLog && v < log_n) return v;
    }
    int k0;
    if (log_n >= 23) k0 = 9;
    else if (log_n >= 14) k0 = log_n - kTileLog;
    else k0 = log_n / 2;
    if (k0 < g) k0 = g;
    if (k0 < 3) k0 = 3;
    return k0;
}

// passes over one row of 2^s0 elements: the last one is a full tile, the first takes the remainder
static int plan_row_passes(int s0, int* ks) {
    if (s0 <= kTileLog) {
        ks[0] = s0;
        return 1;
    }
    int np = 0, rem = s0;
    int tmp[4];
    while (rem > kTileLog) {
        tmp[np++] = kTileLog;
        rem -= kTileLog;
    }
    tmp[np++] = rem;
    for (int i = 0; i < np; i++) ks[i] = tmp[np - 1 - i];
    return np;
}

int ntt_run_sharded(zkr_ctx* ctx, cudaStream_t st, Fr* src, const NttXchg& x, int log_n, bool dit, bool inverse,
                    int (*barrier)(void*, cudaStream_t), void* barrier_arg) {
    NttTables* t;
    ZKR_TRY(ntt_get_tables(ctx, log_n, &t));
    const int g = x.g, k0 = x.k0, s0 = x.s0;
    if (k0 != ntt_sharded_k0(log_n, g) || s0 != log_n - k0 || k0 < 3 || k0 > kTileLog || s0 - g < kTileLog - k0 ||
        s0 < 3 || s0 > 3 * kTileLog) {
        set_error("sharded NTT: 2^%d over 2^%d ranks is too small (or the geometry is inconsistent)", log_n, g);
        return ZKR_E_UNSUPPORTED;
    }
    int ks[4];
    const int np1 = plan_row_passes(s0, ks);      // passes over the columns of one row (local, contiguous rows)
    const double units = (double)((size_t)1 << (log_n - g));
    Fr* dst = x.peer[x.rank];
    PassGeom g0;                                  // the strided pass over the rows, on a COLS slab
    g0.k = k0;
    g0.c = kTileLog - k0;
    g0.s = s0;
    g0.ls = s0 - g;
    g0.chunk_log = 0;
    g0.ctw = (unsigned)x.rank << (s0 - g);
    g0.tw_shift = 0;
    g0.blocks = 1u << (s0 - g - g0.c);
    auto local_geom = [&](int i) {                // pass i (0-based) over the 2^(k0-g) local rows of 2^s0 columns
        PassGeom q;
        q.chunk_log = s0;
        for (int j = 0; j < i; j++) q.chunk_log -= ks[j];
        q.k = ks[i];
        q.s = q.chunk_log - q.k;
        q.c = kTileLog - q.k;
        if (q.c > q.s) q.c = q.s;
        q.ls = q.s;
        q.ctw = 0;
        q.tw_shift = log_n - q.chunk_log;
        q.blocks = 1u << (log_n - g - q.k - q.c);
        return q;
    };
    if (!dit) {
        ZKR_TRY(barrier(barrier_arg, st));        // every rank is done with its destination buffer
        ZKR_TRY(launch_pass<1>(ctx, st, t, src, g0, false, inverse, x, units));
        ZKR_TRY(barrier(barrier_arg, st));        // all remote stores have landed
        for (int i = 0; i < np1; i++) ZKR_TRY(launch_pass<0>(ctx, st, t, dst, local_geom(i), false, inverse, x, units));
    } else {
        for (int i = np1 - 1; i >= 1; i--) ZKR_TRY(launch_pass<0>(ctx, st, t, src, local_geom(i), true, inverse, x, units));
        ZKR_TRY(barrier(barrier_arg, st));
        ZKR_TRY(launch_pass<2>(ctx, st, t, src, local_geom(0), true, inverse, x, units));
        ZKR_TRY(barrier(barrier_arg, st));
        ZKR_TRY(launch_pass<3>(ctx, st, t, dst, g0, true, inverse, x, units));
    }
    return ZKR_OK;
}

int ntt_scale_pow_sharded(zkr_ctx* ctx, cudaStream_t st, Fr* x, const NttXchg& g, int log_n, int layout,
                          const Fr* lo, const Fr* hi, int lb) {
    const size_t nl = (size_t)1 << (log_n - g.g);
    ZKR_LAUNCH(ctx, k_scale_pow_sharded, ceil_div(nl, 128), 128, 0, st, x, nl, log_n, lo, hi, lb, layout, g.s0, g.g, g.rank);
    return ZKR_OK;
}

int ntt_scale_const(zkr_ctx* ctx, cudaStream_t st, Fr* x, size_t n, const Fr* cst) {
    ZKR_LAUNCH(ctx, k_scale_const, ceil_div(n, 128), 128, 0, st, x, n, cst);
    return ZKR_OK;
}

// h = U where A*B = L + x^m U  (SURVEY.md B.4 method iv; oracle: calc_h_lu).
//   S = A_T . B_T            -> DIF^-1 -> m (L+U)_j           at bit-reversed positions
//   a, b = DIF^-1(A_T, B_T)  -> * g^j/m -> DIT -> A, B on the coset g<omega>  (natural order)
//   P = A . B                -> DIF^-1 -> m (L-U)_j g^j
//   h_j = ((L+U)_j - (L-U)_j) / 2
// Pointwise products of two data vectors pick up a factor 1/R (Montgomery); the final constants
// carry R/(2m) so the output has the same form (standard or Montgomery) as the inputs.
//
// No element-wise sweep runs on its own (bit-reversed output, the prover's case): S and P are formed while the first
// pass of their transform loads its tile (LD_MUL2), the coset scaling g^j / m is a table multiply in the load of the DIT
// transforms' first pass (LD_TAB), and h is assembled in the store of the last pass (ST_HFINAL).  A single-pass transform
// (m <= 2^11) would need both LD_MUL2's and ST_HFINAL's second operand in one launch: there P is formed by the sweep.
int h_pipeline(zkr_ctx* ctx, cudaStream_t st, Fr* A, Fr* B, Fr* S, Fr* h, int log_m, bool bitrev_out) {
    NttTables* t;
    ZKR_TRY(ntt_get_tables(ctx, log_m, &t));
    const size_t m = (size_t)1 << log_m;
    const int blk = 128, grid = ceil_div(m, blk);
    static const bool unfused = getenv("ZKR_H_UNFUSED") && atoi(getenv("ZKR_H_UNFUSED")) != 0;   // A/B knob: round-1 pipeline
    if (log_m >= 3 && bitrev_out && !unfused) {
        if (!t->cs_br) {      // cold path: the two position-ordered tables of this size
            ZKR_CUDA(cudaMalloc(&t->cs_br, m * sizeof(Fr)));
            ZKR_CUDA(cudaMalloc(&t->hf_br, m * sizeof(Fr)));
            t->bytes += 2 * m * sizeof(Fr);
            ZKR_LAUNCH(ctx, k_pow_bitrev, ceil_div(m, 256), 256, 0, st, t->cs_br, log_m, t->cs_lo, t->cs_hi_n, t->lb);
            ZKR_LAUNCH(ctx, k_pow_bitrev, ceil_div(m, 256), 256, 0, st, t->hf_br, log_m, t->ci_lo, t->ci_hi_h, t->lb);
        }
        int ks[4];
        const bool single = plan_passes(log_m, ks) == 1;
        PassFuse mulAB = {};
        mulAB.ld_op = LD_MUL2;
        mulAB.src = A;
        mulAB.in2 = B;
        ZKR_TRY(ntt_run_ex(ctx, st, S, log_m, false, true, &mulAB, nullptr));     // S <- DIF^-1(A_T . B_T)
        ZKR_TRY(ntt_run_ex(ctx, st, A, log_m, false, true, nullptr, nullptr, B));  // A and B share every launch
        PassFuse coset = {};
        coset.ld_op = LD_TAB;
        coset.tab = t->cs_br;
        ZKR_TRY(ntt_run_ex(ctx, st, A, log_m, true, false, &coset, nullptr, B));  // A, B on the coset g<omega>
        PassFuse mulP = {}, fin = {};
        mulP.ld_op = LD_MUL2;
        mulP.in2 = B;
        fin.st_op = ST_HFINAL;
        fin.in2 = S;
        fin.tab = t->hf_br;
        fin.kconst = &t->roots->hconst;
        fin.out = h;
        if (single) ZKR_LAUNCH(ctx, k_pointwise_mul, grid, blk, 0, st, A, A, B, m);
        ZKR_TRY(ntt_run_ex(ctx, st, A, log_m, false, true, single ? nullptr : &mulP, &fin));
        return ZKR_OK;
    }
    ZKR_LAUNCH(ctx, k_pointwise_mul, grid, blk, 0, st, S, A, B, m);
    ZKR_TRY(ntt_run(ctx, st, A, log_m, false, true));
    ZKR_TRY(ntt_run(ctx, st, B, log_m, false, true));
    ZKR_TRY(ntt_run(ctx, st, S, log_m, false, true));
    ZKR_LAUNCH(ctx, k_scale_pow, grid, blk, 0, st, A, m, log_m, t->cs_lo, t->cs_hi_n, t->lb, true);
    ZKR_LAUNCH(ctx, k_scale_pow, grid, blk, 0, st, B, m, log_m, t->cs_lo, t->cs_hi_n, t->lb, true);
    ZKR_TRY(ntt_run(ctx, st, A, log_m, true, false));
    ZKR_TRY(ntt_run(ctx, st, B, log_m, true, false));
    ZKR_LAUNCH(ctx, k_pointwise_mul, grid, blk, 0, st, A, A, B, m);
    ZKR_TRY(ntt_run(ctx, st, A, log_m, false, true));
    ZKR_LAUNCH(ctx, k_h_final, grid, blk, 0, st, h, S, A, m, log_m, &t->roots->hconst, t->ci_lo, t->ci_hi_h,
               t->lb, bitrev_out);
    return ZKR_OK;
}

}  // namespace zkr

using namespace zkr;

extern "C" int zkr_ntt(zkr_ctx* ctx, void* data, int log_n, int mode, int on_device) {
    if (!ctx || !data || log_n < 1) return ZKR_E_INVALID;
    const int base_mode = mode & 0xf;
    const bool br_out = mode & ZKR_NTT_BITREV_OUT, br_in = mode & ZKR_NTT_BITREV_IN;
    if (base_mode > 3 || (br_out && br_in)) return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    NttTables* t;
    ZKR_TRY(ntt_get_tables(ctx, log_n, &t));
    const size_t n = (size_t)1 << log_n, bytes = n * sizeof(Fr);
    cudaStream_t st = ctx->user_stream;
    Fr* d = (Fr*)data;
    if (!on_device) {
        void* p;
        ZKR_TRY(ctx->scratch_get("ntt_io", bytes, &p));
        d = (Fr*)p;
        ZKR_CUDA(cudaMemcpyAsync(d, data, bytes, cudaMemcpyHostToDevice, st));
    }
    const bool inverse = base_mode == ZKR_NTT_INVERSE || base_mode == ZKR_NTT_COSET_INVERSE;
    const bool coset = base_mode >= ZKR_NTT_COSET_FORWARD;
    const int blk = 128, grid = ceil_div(n, blk);
    if (coset && !inverse)   // x_j *= g^j, j = natural coefficient index
        ZKR_LAUNCH(ctx, k_scale_pow, grid, blk, 0, st, d, n, log_n, t->cs_lo, t->cs_hi, t->lb, br_in);
    ZKR_TRY(ntt_run(ctx, st, d, log_n, br_in, inverse));
    const bool out_is_bitrev = !br_in;   // DIF leaves bit-reversed order
    if (br_out || br_in) {
        // stay in the order the transform produced; apply the inverse scalings in place
        if (inverse && coset)
            ZKR_LAUNCH(ctx, k_scale_pow, grid, blk, 0, st, d, n, log_n, t->ci_lo, t->ci_hi_n, t->lb, out_is_bitrev);
        else if (inverse)
            ZKR_LAUNCH(ctx, k_scale_const, grid, blk, 0, st, d, n, &t->roots->ninv);
    } else {
        void* p;
        ZKR_TRY(ctx->scratch_get("ntt_tmp", bytes, &p));
        Fr* tmp = (Fr*)p;
        const Fr* cst = inverse && !coset ? &t->roots->ninv : nullptr;
        const Fr* lo = inverse && coset ? t->ci_lo : nullptr;
        ZKR_LAUNCH(ctx, k_bitrev_scale, grid, blk, 0, st, tmp, d, n, log_n, cst, lo, t->ci_hi_n, t->lb);
        ZKR_CUDA(cudaMemcpyAsync(d, tmp, bytes, cudaMemcpyDeviceToDevice, st));
    }
    if (!on_device) {
        ZKR_CUDA(cudaMemcpyAsync(data, d, bytes, cudaMemcpyDeviceToHost, st));
        ZKR_CUDA(cudaStreamSynchronize(st));
    }
    return ZKR_OK;
}

extern "C" int zkr_fill_geometric(zkr_ctx* ctx, void* d_out, size_t n_local, const void* c32, const void* g32,
                                  uint64_t start, int log_n, int world, int rank) {
    if (!ctx || !d_out || !c32 || !g32 || world < 1 || (world & (world - 1)) || rank < 0 || rank >= world) return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->user_stream;
    void* p;
    ZKR_TRY(ctx->scratch_get("fill_cg", 64, &p));
    char cg[64];
    memcpy(cg, c32, 32);
    memcpy(cg + 32, g32, 32);
    ZKR_CUDA(cudaMemcpyAsync(p, cg, 64, cudaMemcpyHostToDevice, st));
    ZKR_CUDA(cudaStreamSynchronize(st));   // cg is a stack buffer
    int wl = -1, s0 = 0;
    if (world > 1) {
        wl = 0;
        while ((1 << wl) < world) wl++;
        s0 = log_n - ntt_sharded_k0(log_n, wl);
        if (log_n < wl || n_local != ((size_t)1 << (log_n - wl)) || s0 < wl) return ZKR_E_INVALID;
    }
    if (n_local)
        ZKR_LAUNCH(ctx, k_fill_geometric, ceil_div(n_local, 128), 128, 0, st, (Fr*)d_out, n_local, (const Fr*)p, start, s0,
                   wl, rank);
    return ZKR_OK;
}

extern "C" int zkr_h_from_evals_dev(zkr_ctx* ctx, void* d_a_t, void* d_b_t, int log_m, void* d_h_out, int bitrev_out) {
    if (!ctx || !d_a_t || !d_b_t || !d_h_out || log_m < 1) return ZKR_E_INVALID;
    DeviceGuard g(ctx->device);
    void* p;
    ZKR_TRY(ctx->scratch_get("h_S", ((size_t)1 << log_m) * sizeof(Fr), &p));
    return h_pipeline(ctx, ctx->user_stream, (Fr*)d_a_t, (Fr*)d_b_t, (Fr*)p, (Fr*)d_h_out, log_m, bitrev_out != 0);
}
