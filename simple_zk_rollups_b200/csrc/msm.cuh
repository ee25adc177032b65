// Signed-digit bucketed Pippenger MSM over precomputed window tables, templated on the curve
// (Fq -> G1, Fq2 -> G2).  Replaces websnark g1_multiexp / g2_multiexp (five calls inside
// groth16GenProof, /root/reference/operator/src/snarks/common.ts:29) and the per-signal
// G1.mulScalar / G2.mulScalar loop of snarkjs prover_groth.js.
//
// B200-first design (DESIGN.md "MSM"):
//   * The bases are static per circuit, HBM is 180 GB: at key-load time every base P_i is expanded
//     to its W window multiples 2^(c w) P_i (affine, Montgomery).  All windows then share ONE set of
//     2^(c-1) buckets, there is no window-combine (no 254 serial doublings), and c can be larger
//     than a per-window scheme allows (c = 17 at n = 2^20 -> 15 mixed adds per point, c = 20 at 2^22 -> 13).
//   * per MSM:  digits (signed, c bits)  ->  radix sort of (bucket, point-ref) pairs  ->
//     chunked bucket accumulation  ->  boundary levels  ->  parallel weighted bucket reduction.
//   * accumulation is perfectly load balanced for ANY scalar distribution: thread t owns entries
//     [tL, (t+1)L) of the bucket-sorted list, adds runs of equal bucket with XYZZ mixed adds, writes
//     complete (interior) runs straight to their bucket and hands its first / last partial run to the
//     next level, which applies the same algorithm to the (<= 2 per thread) boundary partials.  A
//     bucket holding 3 % of all points (the {0,1} witness skew of the rollup circuit) simply spans
//     many threads.
//   * reduction sum_b (b+1) B_b without a serial running sum: row / column sums of the bucket array viewed as a
//     2^lr x 2^lc matrix, then bit-decomposed weighted sums (k_bucket_sums / k_bucket_weighted below).
//   * measured dead ends: capping the G2 accumulation kernel at 168 / 128 registers (3 / 4 CTAs per SM instead of 2,
//     ~90 / ~270 spilled words per addition) makes the 2^20 proof slower, 17.8 / 18.3 ms against 17.3 ms; keeping the
//     accumulator's ZZ / ZZZ in shared memory by hand (168 registers, no spills) is slower too, 17.66 against 16.98 ms
//     (profiles/r02_g2_smem_acc_ab.json; that kernel was deleted); so is splitting every G2 addition over a lane pair
//     with one dual multiplication + one reduction per lane (126 registers, 4 CTAs / SM): 17.09 against 16.94 ms
//     (profiles/r02_g2_pair_lanes_ab.json; deleted as well).
#pragma once
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "ec.cuh"
#include "msm_iface.cuh"

namespace zkr {

constexpr int kAccumThreads = 128;
// Which groups accumulate with XYZZ::madd_lazy (bit 0 G1, bit 1 G2) and whether G1 squares with mont_sqr_raw (bit 2);
// ZKR_LAZY overrides (A/B knob).  Measured on a B200 (profiles/r02_lazy_reduction_ab.json, r02_fast_sqr_ab.json): G1 launch
// 1.91 -> 1.80 -> 1.73 ms, 2^20 proof 16.79 -> 15.34 -> 15.08 ms.
constexpr int kLazyDefault = 7;
constexpr int kLevelLog = 4;          // boundary levels: 16 entries per thread ...
constexpr int kLevelLogBig = 2;       // ... except while the list is long: 4 per thread keeps ~4x more warps in flight
constexpr size_t kLevelBigMin = 1u << 16;
inline int level_log(size_t cnt) { return cnt >= kLevelBigMin ? kLevelLogBig : kLevelLog; }
constexpr uint32_t kNegBit = 0x80000000u;
// Zero digits carry the sentinel key 2^(c-1): they sort behind every bucket and the accumulation kernel never visits
// them.  Folding them into the buckets as "skip" entries saves a key bit (two radix passes instead of three at c = 17)
// but makes the IMAD-bound accumulation loop visit 3 % more entries: measured slower (profiles/r02_zero_digit_sort_ab.json).

struct MsmPlan {
    int c = 0, W = 0;
    uint32_t nbuckets = 0;            // 2^(c-1); also the sentinel key of skipped (zero) digits
    static MsmPlan choose(uint64_t n, int c_forced) {
        MsmPlan p;
        int best = 0;
        double best_cost = 1e300;
        for (int c = 4; c <= 23; c++) {
            int W = (255 + c - 1) / c;
            if ((uint64_t)W * n >= (1ull << 31)) continue;
            double cost = 10.0 * (double)n * W + 56.0 * (double)(1u << (c - 1));
            if (cost < best_cost) { best_cost = cost; best = c; }
        }
        if (c_forced <= 0)
            if (const char* e = getenv("ZKR_MSM_C")) c_forced = atoi(e);      // A/B knob (profiles/r02_window_sweep.json)
        if (c_forced > 0 && (uint64_t)((255 + c_forced - 1) / c_forced) * n >= (1ull << 31)) c_forced = 0;
        p.c = c_forced > 0 ? c_forced : best;
        p.W = (255 + p.c - 1) / p.c;
        p.nbuckets = 1u << (p.c - 1);
        return p;
    }
};

// ------------------------------------------------------------------------------------------------
// table[w * n + i] = 2^(c w) * P_i, affine Montgomery
template <class F>
__global__ void k_precompute(const char* __restrict__ pts, char* __restrict__ table, uint32_t n, int c, int W) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    constexpr size_t AB = 2 * sizeof(F);
    Affine<F> p = Affine<F>::load(pts + AB * i);
    p.store(table + AB * i);
    XYZZ<F> acc = XYZZ<F>::from_affine(p);
    for (int w = 1; w < W; w++) {
#pragma unroll 1
        for (int d = 0; d < c; d++) acc = acc.dbl();
        Affine<F> a = acc.to_affine();
        a.store(table + AB * ((size_t)w * n + i));
    }
}

// keys[w n + i] = kofs + |digit| - 1 (or sentinel for 0), vals[w n + i] = (w n + i) | sign
__device__ __forceinline__ void scalar_digits(const Fr& k, uint32_t i, uint32_t n, int c, int W, uint32_t kofs,
                                              uint32_t sentinel, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint32_t carry = 0;
    const uint32_t half = 1u << (c - 1), mask = (1u << c) - 1;
    for (int w = 0; w < W; w++) {
        int bit = w * c, limb = bit >> 5, sh = bit & 31;
        uint32_t d = 0;
        if (limb < 8) {
            d = k.v[limb] >> sh;
            if (sh + c > 32 && limb + 1 < 8) d |= k.v[limb + 1] << (32 - sh);
        }
        d = (d & mask) + carry;
        uint32_t neg = 0;
        carry = 0;
        if (d > half) {
            d = (1u << c) - d;
            neg = kNegBit;
            carry = 1;
        }
        uint32_t pos = (uint32_t)w * n + i;
        // a zero digit gets the sentinel key: it sorts behind every bucket and the accumulation never visits it (see kNegBit)
        keys[pos] = d ? kofs + d - 1 : sentinel;
        vals[pos] = pos | neg;
    }
}

static __global__ void k_digits(const uint32_t* __restrict__ scalars, const uint32_t* __restrict__ src_index, uint32_t n,
                         int c, int W, uint32_t sentinel, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                         int* __restrict__ range_err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* sp = scalars + 8 * (size_t)(src_index ? src_index[i] : i);
    Fr k = Fr::load_ro(sp);
    if (!k.in_range()) *range_err = 1;
    scalar_digits(k, i, n, c, W, 0, sentinel, keys, vals);
}

// Batched form (msm_run_many): vector j = blockIdx.y is read at scalars + 8 stride j and owns the entries
// [j W n, (j+1) W n) and the buckets [j nb, (j+1) nb); the table reference in vals is the same for every vector.
static __global__ void k_digits_many(const uint32_t* __restrict__ scalars, size_t stride, const uint32_t* __restrict__ src_index,
                                     uint32_t n, int c, int W, uint32_t nb, uint32_t sentinel, uint32_t* __restrict__ keys,
                                     uint32_t* __restrict__ vals, int* __restrict__ range_err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= n) return;
    const uint32_t* sp = scalars + 8 * (stride * j + (src_index ? src_index[i] : i));
    Fr k = Fr::load_ro(sp);
    if (!k.in_range()) range_err[j] = 1;
    const size_t base = (size_t)j * W * n;
    scalar_digits(k, i, n, c, W, j * nb, sentinel, keys + base, vals + base);
}

// ------------------------------------------------------------------------------------------------
// level 1: affine table entries -> bucket sums / boundary partials
// It also records where every bucket's run begins and ends in the sorted list (run_lo / run_hi, null = off): the thread
// that sees a key change owns that boundary; the boundary at a chunk's first entry is found by reading the previous
// chunk's last key.  k_bucket_gather turns the head / tail partials into bucket sums with these bounds in ONE launch.
// LAZY: the mixed addition with sums of products reduced once (XYZZ::madd_lazy; same words out).
template <class F, bool PREFETCH, int LAZY>      // LAZY 2: madd_lazy with the dedicated squaring (fp.cuh mont_sqr_raw)
__global__ void __launch_bounds__(kAccumThreads, sizeof(F) == 32 ? 4 : 2)       // G1: 128 registers, 4 CTAs / SM
k_accum_affine(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t total, int logL,
               const char* __restrict__ table, XYZZ<F>* __restrict__ buckets, XYZZ<F>* __restrict__ bnd,
               uint32_t* __restrict__ bnd_keys, uint32_t sentinel, uint32_t* __restrict__ run_lo) {
    uint32_t* const run_hi = run_lo + sentinel;      // one allocation: [lo of every bucket | hi of every bucket]
    extern __shared__ uint32_t sm[];
    constexpr size_t AB = 2 * sizeof(F);
    const int L = 1 << logL, LP = L + 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* sk = sm + warp * 2 * 32 * LP;
    uint32_t* sv = sk + 32 * LP;
    const size_t wchunk = (size_t)blockIdx.x * (kAccumThreads / 32) + warp;   // warp-sized group of chunks
    const size_t wbase = wchunk * 32 * L;
    for (int i = lane; i < 32 * L; i += 32) {
        size_t e = wbase + i;
        uint32_t kk = sentinel, vv = 0;
        if (e < total) {
            kk = keys[e];
            vv = vals[e];
        }
        int r = i >> logL, ci = i & (L - 1);
        sk[r * LP + ci] = kk;
        sv[r * LP + ci] = vv;
    }
    __syncwarp();
    const uint32_t* mk = sk + lane * LP;
    const uint32_t* mv = sv + lane * LP;
    const size_t t = wchunk * 32 + lane;

    XYZZ<F> acc = XYZZ<F>::identity();
    uint32_t cur = mk[0];
    bool first_run = true;
    uint32_t head_key = sentinel, tail_key = sentinel;
    Affine<F> nxt;
    bool have = cur < sentinel;
    const uint32_t p0 = (uint32_t)t << logL;         // sorted position of this chunk's first entry (< 2^31 + padding)
    if (run_lo && p0 <= total) {
        const uint32_t prevk = (p0 > 0) ? keys[p0 - 1] : sentinel;
        if (p0 == 0 || prevk != cur) {
            if (have) run_lo[cur] = p0;
            if (p0 > 0 && prevk < sentinel) run_hi[prevk] = p0;
        }
    }
    if (PREFETCH && have) nxt = Affine<F>::load_ro(table + AB * (size_t)(mv[0] & ~kNegBit));
    int j = 0;                                       // after the loop: the chunk's first unprocessed entry (a sentinel) or L
    for (; j < L; j++) {
        if (!have) break;
        const uint32_t key = mk[j], v = mv[j];
        Affine<F> p;
        if (PREFETCH) p = nxt;
        else p = Affine<F>::load_ro(table + AB * (size_t)(v & ~kNegBit));
        have = (j + 1 < L) && (mk[j + 1] < sentinel);
        if (PREFETCH && have) nxt = Affine<F>::load_ro(table + AB * (size_t)(mv[j + 1] & ~kNegBit));
        if (key != cur) {
            if (run_lo) {
                run_hi[cur] = p0 + j;
                run_lo[key] = p0 + j;
            }
            if (first_run) {
                acc.store(bnd + 2 * t);
                head_key = cur;
                first_run = false;
            } else {
                acc.store(buckets + cur);
            }
            acc = XYZZ<F>::identity();
            cur = key;
        }
        if (v & kNegBit) p.y = p.y.neg();
        if (LAZY == 2) acc.template madd_lazy<true>(p);
        else if (LAZY == 1) acc.template madd_lazy<false>(p);
        else acc.madd(p);
    }
    if (cur < sentinel) {
        if (first_run) {
            acc.store(bnd + 2 * t);
            head_key = cur;
        } else {
            acc.store(bnd + 2 * t + 1);
            tail_key = cur;
        }
        if (run_lo) {
            // the run's end, if it lies in this chunk: a sentinel follows, or the list ends at / before the chunk's end
            // (the boundary at the next chunk's first entry belongs to that chunk's thread)
            if (j < L) run_hi[cur] = p0 + j;
            else if (p0 + L >= total) run_hi[cur] = total;
        }
    }
    if (bnd_keys) {
        bnd_keys[2 * t] = head_key;
        bnd_keys[2 * t + 1] = tail_key;
    }
}

// ------------------------------------------------------------------------------------------------
// Boundary partials -> bucket sums in ONE launch (replaces the recursive boundary levels + k_accum_finish: up to 7
// launches of shrinking, latency-bound work per MSM).  Bucket b's entries are the sorted positions [lo, hi); level-1
// thread t owns [t L, (t+1) L).  The partial sums of b are therefore
//     thread t0 = lo / L : its HEAD slot if the run starts the chunk, else its TAIL slot -- unless the run lies strictly
//                          inside the chunk, in which case level 1 has already stored the complete bucket;
//     threads t0+1 .. t1 = (hi-1) / L : their HEAD slots (the run starts their chunk).
// One thread per bucket adds them (about run length / L + 1 additions: ~7 at 2^20); buckets with more than kHeavyRun
// partials (the {0, 1} witness skew, adversarial scalar sets) are summed by whole CTAs of the same launch.
constexpr int kGatherThreads = 128;
constexpr uint32_t kHeavyRun = 48;
constexpr uint32_t kNoRun = 0xffffffffu;
constexpr int kHeavyBlocks = 64;

// Blocks [0, kHeavyBlocks) are the heavy path, launched first so that their few long chains run beside the light
// blocks of the same launch: the heavy blocks scan the run bounds (bucket b belongs to heavy block b mod kHeavyBlocks) and
// sum each bucket that has more than kHeavyRun partials with all their threads (strided partial sums, then a tree in
// shared memory).
// Blocks [kHeavyBlocks, ...) are the light path: one thread per bucket.
template <class F>
__global__ void __launch_bounds__(kGatherThreads)
k_bucket_gather(const uint32_t* __restrict__ keys, uint32_t total, int logL, const uint32_t* __restrict__ run_lo,
                const XYZZ<F>* __restrict__ bnd, XYZZ<F>* __restrict__ buckets, uint32_t nbuckets) {
    extern __shared__ unsigned char smraw[];
    const uint32_t* run_hi = run_lo + nbuckets;
    if (blockIdx.x < kHeavyBlocks) {
        XYZZ<F>* sp = reinterpret_cast<XYZZ<F>*>(smraw);
        __shared__ uint32_t found[kGatherThreads];
        __shared__ uint32_t n_found;
        for (uint32_t b0 = blockIdx.x; b0 < nbuckets; b0 += kHeavyBlocks * kGatherThreads) {
            // heavy block h owns the buckets b = h (mod kHeavyBlocks): neighbouring heavy buckets (small digits of a short
            // top window, adversarial scalar sets) land on different blocks.  Most iterations find none: one barrier.
            // The scan is cheap; what costs is ~50 us of whole-CTA work per heavy bucket -- 4096 of them at 22-bit windows
            // (2^24 points: the 12-bit top window) made this kernel 9 ms, one reason the recursive levels serve c > 20.
            const uint32_t b = b0 + threadIdx.x * kHeavyBlocks;
            bool is_heavy = false;
            if (b < nbuckets) {
                const uint32_t lo = run_lo[b];
                is_heavy = lo != kNoRun && (((run_hi[b] - 1) >> logL) - (lo >> logL) + 1) > kHeavyRun;
            }
            if (__syncthreads_count(is_heavy) == 0) continue;
            if (threadIdx.x == 0) n_found = 0;
            __syncthreads();
            if (is_heavy) found[atomicAdd(&n_found, 1u)] = b;
            __syncthreads();
            const uint32_t nf = n_found;
            for (uint32_t f = 0; f < nf; f++) {
                const uint32_t hb = found[f];
                const uint32_t lo = run_lo[hb], hi = run_hi[hb];
                const uint32_t t0 = lo >> logL, t1 = (hi - 1) >> logL;
                const bool aligned = lo == (t0 << logL);
                XYZZ<F> acc = XYZZ<F>::identity();
#pragma unroll 1
                for (uint32_t t = t0 + threadIdx.x; t <= t1; t += kGatherThreads)
                    acc.add(XYZZ<F>::load(bnd + 2 * (size_t)t + ((t == t0 && !aligned) ? 1 : 0)));
                sp[threadIdx.x] = acc;
                __syncthreads();
                for (int d = kGatherThreads / 2; d >= 1; d >>= 1) {
                    if ((int)threadIdx.x < d) xyzz_add_mem(&sp[threadIdx.x], &sp[threadIdx.x], &sp[threadIdx.x + d]);
                    __syncthreads();
                }
                if (threadIdx.x == 0) sp[0].store(buckets + hb);
                __syncthreads();
            }
            __syncthreads();
        }
        return;
    }
    const uint32_t b = (blockIdx.x - kHeavyBlocks) * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    const uint32_t lo = run_lo[b];
    if (lo == kNoRun) return;                         // empty bucket: stays the identity (memset)
    const uint32_t hi = run_hi[b];
    const uint32_t t0 = lo >> logL, t1 = (hi - 1) >> logL;
    const bool aligned = lo == (t0 << logL);
    if (t0 == t1) {
        // one chunk: head slot, tail slot (run reaches the chunk's end or the end of the real entries), or already complete
        const bool to_end = hi >= ((t0 + 1) << logL) || hi >= total || keys[hi] >= nbuckets;
        if (aligned) XYZZ<F>::load(bnd + 2 * (size_t)t0).store(buckets + b);
        else if (to_end) XYZZ<F>::load(bnd + 2 * (size_t)t0 + 1).store(buckets + b);
        return;
    }
    if (t1 - t0 + 1 > kHeavyRun) return;              // summed by a heavy block of this launch
    XYZZ<F> acc = XYZZ<F>::load(bnd + 2 * (size_t)t0 + (aligned ? 0 : 1));
#pragma unroll 1
    for (uint32_t t = t0 + 1; t <= t1; t++) acc.add(XYZZ<F>::load(bnd + 2 * (size_t)t));
    acc.store(buckets + b);
}

// level >= 2: XYZZ partials (with sentinel holes) -> bucket sums / boundary partials
template <class F>
__global__ void __launch_bounds__(64)
k_accum_xyzz(const uint32_t* __restrict__ in_keys, const XYZZ<F>* __restrict__ in_pts, uint32_t count, int logL,
             XYZZ<F>* __restrict__ buckets, XYZZ<F>* __restrict__ bnd, uint32_t* __restrict__ bnd_keys,
             uint32_t sentinel, bool final_level) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t begin = t << logL;
    if (begin >= count) {
        if (!final_level) {
            // threads past the end still own boundary slots the next level will read
            bnd_keys[2 * t] = sentinel;
            bnd_keys[2 * t + 1] = sentinel;
        }
        return;
    }
    size_t end = begin + ((size_t)1 << logL);
    if (end > count) end = count;
    XYZZ<F> acc = XYZZ<F>::identity();
    uint32_t cur = sentinel;
    bool first_run = true;
    uint32_t head_key = sentinel, tail_key = sentinel;
    for (size_t e = begin; e < end; e++) {
        const uint32_t key = in_keys[e];
        if (key >= sentinel) continue;
        if (cur == sentinel) cur = key;
        if (key != cur) {
            if (first_run && !final_level) {
                acc.store(bnd + 2 * t);
                head_key = cur;
            } else {
                acc.store(buckets + cur);
            }
            first_run = false;
            acc = XYZZ<F>::identity();
            cur = key;
        }
        acc.add(XYZZ<F>::load(in_pts + e));
    }
    if (cur < sentinel) {
        if (final_level) {
            acc.store(buckets + cur);
        } else if (first_run) {
            acc.store(bnd + 2 * t);
            head_key = cur;
        } else {
            acc.store(bnd + 2 * t + 1);
            tail_key = cur;
        }
    }
    if (!final_level) {
        bnd_keys[2 * t] = head_key;
        bnd_keys[2 * t + 1] = tail_key;
    }
}

// all remaining boundary levels in ONE launch (single CTA): used once the list is short enough that
// launch latency, not work, dominates.  Buffers ping-pong in global memory; __syncthreads orders them.
constexpr int kFinishThreads = 256;
constexpr uint32_t kFinishMax = kFinishThreads << kLevelLog;      // 4096 entries
template <class F>
__global__ void __launch_bounds__(kFinishThreads)
k_accum_finish(uint32_t* keys_a, XYZZ<F>* pts_a, uint32_t* keys_b, XYZZ<F>* pts_b, uint32_t count,
               XYZZ<F>* __restrict__ buckets, uint32_t sentinel) {
    const uint32_t t = threadIdx.x;
    uint32_t* in_keys = keys_a;
    XYZZ<F>* in_pts = pts_a;
    uint32_t* out_keys = keys_b;
    XYZZ<F>* out_pts = pts_b;
    for (;;) {
        const bool final_level = count <= (1u << kLevelLog);
        const uint32_t T = (count + (1u << kLevelLog) - 1) >> kLevelLog;
        if (t < T) {
            const uint32_t begin = t << kLevelLog;
            uint32_t end = begin + (1u << kLevelLog);
            if (end > count) end = count;
            XYZZ<F> acc = XYZZ<F>::identity();
            uint32_t cur = sentinel, head_key = sentinel, tail_key = sentinel;
            bool first_run = true;
#pragma unroll 1
            for (uint32_t e = begin; e < end; e++) {
                const uint32_t key = in_keys[e];
                if (key >= sentinel) continue;
                if (cur == sentinel) cur = key;
                if (key != cur) {
                    if (first_run && !final_level) {
                        acc.store(out_pts + 2 * t);
                        head_key = cur;
                    } else {
                        acc.store(buckets + cur);
                    }
                    first_run = false;
                    acc = XYZZ<F>::identity();
                    cur = key;
                }
                acc.add(XYZZ<F>::load(in_pts + e));
            }
            if (cur < sentinel) {
                if (final_level) {
                    acc.store(buckets + cur);
                } else if (first_run) {
                    acc.store(out_pts + 2 * t);
                    head_key = cur;
                } else {
                    acc.store(out_pts + 2 * t + 1);
                    tail_key = cur;
                }
            }
            if (!final_level) {
                out_keys[2 * t] = head_key;
                out_keys[2 * t + 1] = tail_key;
            }
        }
        if (final_level) break;
        __syncthreads();
        count = 2 * T;
        uint32_t* tk = in_keys; in_keys = out_keys; out_keys = tk;
        XYZZ<F>* tp = in_pts; in_pts = out_pts; out_pts = tp;
    }
}

// ------------------------------------------------------------------------------------------------
// block-wide helpers on XYZZ points staged in shared memory (blockDim.x == NT, power of two).
// All point arithmetic goes through the memory-to-memory helpers of ec.cuh.
// sum of sp[0..NT) -> sp[0]
template <class F, int NT>
__device__ __forceinline__ void block_sum_inplace(XYZZ<F>* sp) {
    const int l = threadIdx.x;
    __syncthreads();
    for (int d = NT / 2; d >= 1; d >>= 1) {
        if (l < d) xyzz_add_mem(&sp[l], &sp[l], &sp[l + d]);
        __syncthreads();
    }
}

// inclusive suffix sums T_l = sum_{l' >= l} v_l' (Hillis-Steele, ping-pong); returns the buffer holding T
template <class F, int NT>
__device__ __forceinline__ XYZZ<F>* block_suffix_scan(XYZZ<F>* cur, XYZZ<F>* nxt) {
    const int l = threadIdx.x;
    __syncthreads();
    for (int d = 1; d < NT; d <<= 1) {
        if (l + d < NT) xyzz_add_mem(&nxt[l], &cur[l], &cur[l + d]);
        else nxt[l] = cur[l];
        __syncthreads();
        XYZZ<F>* t = cur;
        cur = nxt;
        nxt = t;
    }
    return cur;
}

// *p = k * *p  (p, tmp in shared memory; single thread)
template <class F>
__device__ __forceinline__ void mul_small_mem(XYZZ<F>* p, XYZZ<F>* tmp, uint32_t k) {
    *tmp = *p;
    *p = XYZZ<F>::identity();
    while (k) {
        if (k & 1) xyzz_add_mem(p, p, tmp);
        k >>= 1;
        if (k) xyzz_dbl_mem(tmp);
    }
}

// One warp per CTA: these kernels are latency chains (tree levels of ~4 us point additions) that run
// beside the other MSMs' bulk kernels; a 256-thread CTA of idle tree threads pins 33-65 K registers of an SM
// (measured: the overlapped proof got 0.8 ms SLOWER with 256-thread reduction CTAs although the serialised
// one got 2.4 ms faster).  32 threads x up to 255 registers leave the SM to the accumulation kernels.
constexpr int kReduceThreads = 32;
// (256-thread CTAs for small MSMs -- one element per thread, 8 tree levels -- were timed in round 2 and are slower
// everywhere: profiles/r02_reduce_width_ab.json.)

// Bucket reduction  sum_b (b+1) B_b  without a serial running sum.  Split b = hi * 2^lc + lo:
//     sum_b b B_b = 2^lc * sum_hi hi * Row[hi]  +  sum_lo lo * Col[lo],      sum_b B_b = sum_hi Row[hi]
// with Row[hi] = sum_lo B[hi, lo] and Col[lo] = sum_hi B[hi, lo] (plain sums: one CTA each, tree-reduced),
// and each weighted sum over <= 2^12 entries by bit decomposition,  sum_i i S_i = sum_j 2^j (sum_{i: bit j} S_i):
// one CTA per bit does a plain masked sum and its doublings; the last CTA to finish adds the <= 24 terms.
// Every bucket is added exactly twice (like the running sum) but every addition is independent, so the
// latency of the reduction is ~2 tree depths + (c-2) doublings instead of thousands of chained additions.

// stage 1: CTA g < 2^lr: Row[g];  CTA 2^lr + l: Col[l]
template <class F, int NT>
__device__ __forceinline__ void bucket_sums(const XYZZ<F>* __restrict__ buckets, int lr, int lc, XYZZ<F>* __restrict__ out) {
    extern __shared__ unsigned char smraw[];
    XYZZ<F>* s0 = reinterpret_cast<XYZZ<F>*>(smraw);
    const uint32_t t = threadIdx.x, g = blockIdx.x;
    const bool row = g < (1u << lr);
    const uint32_t len = row ? (1u << lc) : (1u << lr);
    const XYZZ<F>* base = row ? buckets + ((size_t)g << lc) : buckets + (g - (1u << lr));
    const size_t stride = row ? 1 : ((size_t)1 << lc);
    if (t < len) s0[t] = base[t * stride];
    else s0[t] = XYZZ<F>::identity();
#pragma unroll 1
    for (uint32_t i = t + NT; i < len; i += NT) xyzz_add_mem(&s0[t], &s0[t], &base[i * stride]);
    block_sum_inplace<F, NT>(s0);
    if (t == 0) out[g] = s0[0];
}
template <class F, int NT>
__global__ void __launch_bounds__(NT)
k_bucket_sums(const XYZZ<F>* __restrict__ buckets, int lr, int lc, XYZZ<F>* __restrict__ out) {
    bucket_sums<F, NT>(buckets, lr, lc, out);
}
// batched: vector blockIdx.y reduces its own nb buckets into its own nred-entry segment of the scratch
template <class F, int NT>
__global__ void __launch_bounds__(NT)
k_bucket_sums_many(const XYZZ<F>* __restrict__ buckets, uint32_t nb, int lr, int lc, XYZZ<F>* __restrict__ red, uint32_t nred) {
    bucket_sums<F, NT>(buckets + (size_t)blockIdx.y * nb, lr, lc, red + (size_t)blockIdx.y * nred);
}

// stage 2: CTA j < lr: 2^(j+lc) * sum_{hi: bit j} Row[hi];  CTA lr + j, j < lc: 2^j * sum_{lo: bit j} Col[lo];
//          CTA lr + lc: sum_hi Row[hi].  terms -> sums[2^lr + 2^lc ..]; the last CTA adds them into *out.
template <class F, int NT>
__device__ __forceinline__ void bucket_weighted(XYZZ<F>* __restrict__ sums, int lr, int lc, unsigned int* __restrict__ counter,
                                                XYZZ<F>* __restrict__ out) {
    extern __shared__ unsigned char smraw[];
    XYZZ<F>* s0 = reinterpret_cast<XYZZ<F>*>(smraw);
    __shared__ bool last;
    const uint32_t t = threadIdx.x;
    const int g = blockIdx.x, nterms = lr + lc + 1;
    const bool row = g < lr || g == lr + lc;
    const int bit = g == lr + lc ? -1 : (g < lr ? g : g - lr);
    const uint32_t len = row ? (1u << lr) : (1u << lc);
    const XYZZ<F>* src = row ? sums : sums + ((size_t)1 << lr);
    XYZZ<F>* terms = sums + ((size_t)1 << lr) + ((size_t)1 << lc);
    s0[t] = XYZZ<F>::identity();
#pragma unroll 1
    for (uint32_t i = t; i < len; i += NT)
        if (bit < 0 || ((i >> bit) & 1)) xyzz_add_mem(&s0[t], &s0[t], &src[i]);
    block_sum_inplace<F, NT>(s0);
    if (t == 0) {
        const int dbl = bit < 0 ? 0 : (g < lr ? bit + lc : bit);
#pragma unroll 1
        for (int d = 0; d < dbl; d++) xyzz_dbl_mem(&s0[0]);
        terms[g] = s0[0];
        __threadfence();
        last = atomicAdd(counter, 1u) == (unsigned)(nterms - 1);
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (t < (uint32_t)nterms) {
        // written by other CTAs of this launch: read through L2
        const uint4* src16 = reinterpret_cast<const uint4*>(terms + t);
        uint4* dst16 = reinterpret_cast<uint4*>(s0 + t);
#pragma unroll
        for (int i = 0; i < (int)(sizeof(XYZZ<F>) / 16); i++) dst16[i] = __ldcg(src16 + i);
    } else {
        s0[t] = XYZZ<F>::identity();
    }
    block_sum_inplace<F, NT>(s0);
    if (t == 0) {
        s0[0].store(out);
        *counter = 0;
    }
}
template <class F, int NT>
__global__ void __launch_bounds__(NT)
k_bucket_weighted(XYZZ<F>* __restrict__ sums, int lr, int lc, unsigned int* __restrict__ counter, XYZZ<F>* __restrict__ out) {
    bucket_weighted<F, NT>(sums, lr, lc, counter, out);
}
// batched: vector blockIdx.y has its own scratch segment and completion counter, and writes its result at out + y out_stride
template <class F, int NT>
__global__ void __launch_bounds__(NT)
k_bucket_weighted_many(XYZZ<F>* __restrict__ red, uint32_t nred, int lr, int lc, unsigned int* __restrict__ counters,
                       char* __restrict__ out, size_t out_stride) {
    const uint32_t j = blockIdx.y;
    bucket_weighted<F, NT>(red + (size_t)j * nred, lr, lc, counters + j, reinterpret_cast<XYZZ<F>*>(out + j * out_stride));
}

// XYZZ (Montgomery) -> affine standard form bytes; identity -> zeros.  One thread at the tail of a standalone MSM:
// the variable-time inversion (fp_inv.cuh) is the whole kernel.
template <class F>
__device__ __forceinline__ void xyzz_to_affine_std(const XYZZ<F>* in, char* out) {
    Affine<F> a = XYZZ<F>::load(in).to_affine_vartime();
    a.x.from_mont().store(out);
    a.y.from_mont().store(out + sizeof(F));
}
template <class F>
__global__ void k_xyzz_to_affine_std(const XYZZ<F>* in, char* out) {
    xyzz_to_affine_std(in, out);
}
// one single-thread block per result of a batch
template <class F>
__global__ void k_xyzz_to_affine_std_many(const XYZZ<F>* in, char* out) {
    xyzz_to_affine_std(in + blockIdx.x, out + 2 * sizeof(F) * blockIdx.x);
}

// ------------------------------------------------------------------------------------------------
struct MsmWork {                      // per-bases device work buffers
    uint32_t *keys[2] = {nullptr, nullptr}, *vals[2] = {nullptr, nullptr};
    void* cub_tmp = nullptr;
    size_t cub_bytes = 0;
    void* buckets = nullptr;
    void* bnd[2] = {nullptr, nullptr};
    uint32_t* bnd_keys[2] = {nullptr, nullptr};
    void* red = nullptr;              // 2^lr + 2^lc row / column sums, then lr + lc + 1 weighted terms
    unsigned int* red_counter = nullptr;
    void* result = nullptr;           // 1 XYZZ
    uint32_t *run_lo = nullptr, *run_hi = nullptr;     // per bucket: [lo, hi) of its run in the sorted list (kNoRun = empty)
    int* range_err = nullptr;
    size_t bytes = 0;
    // where the last radix sort left the sorted (bucket, point-ref) pairs: read by a second base set that shares them
    mutable const uint32_t* sorted_keys = nullptr;
    mutable const uint32_t* sorted_vals = nullptr;
};

// Optional hooks of one msm_run call (prover.cu).
//   sorted_from : skip digit extraction and the radix sort and consume the sorted pairs another base set (same
//                 scalars, same compaction map, same window plan: pi_b's B2' for B1') produced in this proof; the
//                 caller has made `st` wait for that set's ev_sorted.
//   ev_sorted   : recorded on st once the sorted pairs are final.
struct MsmHooks {
    const zkr_bases* sorted_from = nullptr;
    cudaEvent_t ev_sorted = nullptr;
};

// Work buffers of msm_run_many: up to `cap` scalar vectors over one base set in one pass (DESIGN.md 4.10).  Vector j's
// digits are keyed j * nbuckets + |digit| - 1, so the k vectors are one MSM over k x W x n entries and k x nbuckets
// buckets; only the bucket reduction has a batch dimension.
struct MsmMany {
    int cap = 0;
    int logL = 3;                     // level-1 entries per thread, fixed by cap (the bnd buffers are sized for it)
    uint32_t T1p = 0;
    uint32_t *keys[2] = {nullptr, nullptr}, *vals[2] = {nullptr, nullptr};   // null: sorts are borrowed (sorted_from)
    void* cub_tmp = nullptr;
    size_t cub_bytes = 0;
    void* buckets = nullptr;          // cap x nbuckets
    void* bnd[2] = {nullptr, nullptr};
    uint32_t* bnd_keys[2] = {nullptr, nullptr};
    void* red = nullptr;              // cap x nred: each vector's row / column sums and weighted terms
    uint32_t nred = 0;
    unsigned int* red_counter = nullptr;   // cap completion counters
    uint32_t* run_lo = nullptr;       // 2 x cap x nbuckets
    int* range_err = nullptr;         // cap flags: vector j has a scalar >= r
    void* result = nullptr;           // cap XYZZ results (zkr_msm_many)
    size_t bytes = 0;
    const uint32_t* sorted_keys = nullptr;
    const uint32_t* sorted_vals = nullptr;
};

}  // namespace zkr

struct zkr_bases {
    zkr_ctx* ctx = nullptr;
    int group = 1;
    uint64_t n_src = 0;               // points handed in (including infinities)
    uint32_t n = 0;                   // after dropping infinities
    uint32_t* src_index = nullptr;    // device, compact -> source index; null if identity
    char* table = nullptr;            // device [W][n] affine Montgomery
    zkr::MsmPlan plan;
    zkr::MsmWork work;
    size_t bytes = 0;
    int logL = 5;
    uint32_t T1p = 0;                 // level-1 threads (padded to whole blocks)
    uint64_t map_hash = 0;            // FNV-1a of the compact -> scalar index map (equal maps <=> shareable sort)
    zkr::MsmMany* many = nullptr;     // zkr_msm_many's work buffers: grown on first use, freed with the bases
};

namespace zkr {

// h_scalar_idx (nullable): for input point i the index of its scalar in the scalar vector handed to
// msm_run (default i).  Used by the prover to splice the blinding terms into the key's base sets.
template <class F>
int bases_build(zkr_ctx* ctx, zkr_bases* b, const char* h_points, size_t n_src, int c_forced, cudaStream_t st,
                const uint32_t* h_scalar_idx = nullptr);
template <class F>
int msm_run(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, const uint32_t* d_scalars, XYZZ<F>* d_out,
            const MsmHooks* hooks = nullptr);
// Batched MSM over one base set: vector j's scalars at d_scalars + 32 * stride * j bytes (through the same compaction
// map), its XYZZ result at (char*)d_out + j * out_stride.  sorted_from: take the sorted pairs of another base set's
// batch of this call (same conditions as MsmHooks::sorted_from); ev_sorted: recorded once this batch's sort is final.
template <class F>
int many_alloc(const zkr_bases* b, int cap, bool sorts, cudaStream_t st, MsmMany* w);
template <class F>
int msm_run_many(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, MsmMany* w, int k, const uint32_t* d_scalars,
                 size_t stride, void* d_out, size_t out_stride, const MsmMany* sorted_from, cudaEvent_t ev_sorted);
void bases_release(zkr_bases* b);

// ---------------------------------------------------------------- implementation (header-only, two TUs)
template <class F>
int bases_build(zkr_ctx* ctx, zkr_bases* b, const char* h_points, size_t n_src, int c_forced, cudaStream_t st,
                const uint32_t* h_scalar_idx) {
    constexpr size_t AB = 2 * sizeof(F);
    constexpr size_t XB = 4 * sizeof(F);
    b->ctx = ctx;
    b->n_src = n_src;
    // host-side compaction: x == 0 (all coordinate bytes zero) marks infinity (binarify.ts:92-95)
    std::vector<uint32_t> idx;
    idx.reserve(n_src);
    for (size_t i = 0; i < n_src; i++) {
        const uint64_t* x = reinterpret_cast<const uint64_t*>(h_points + AB * i);
        uint64_t any = 0;
        for (size_t j = 0; j < sizeof(F) / 8; j++) any |= x[j];
        if (any) idx.push_back((uint32_t)i);
    }
    b->n = (uint32_t)idx.size();
    const uint32_t n = b->n;
    {
        uint64_t h = 1469598103934665603ull;
        for (uint32_t k = 0; k < n; k++) {
            const uint32_t v = h_scalar_idx ? h_scalar_idx[idx[k]] : idx[k];
            for (int sft = 0; sft < 32; sft += 8) h = (h ^ ((v >> sft) & 0xff)) * 1099511628211ull;
        }
        b->map_hash = h;
    }
    b->plan = MsmPlan::choose(n ? n : 1, c_forced);
    const int W = b->plan.W;
    if ((uint64_t)W * n >= (1ull << 31)) {
        set_error("MSM too large: %u points x %d windows exceeds 2^31 entries", n, W);
        return ZKR_E_UNSUPPORTED;
    }
    if (n == 0) return ZKR_OK;
    char* d_pts = nullptr;
    ZKR_CUDA(cudaMalloc(&d_pts, AB * (size_t)n));
    if (n == n_src && !h_scalar_idx) {
        ZKR_CUDA(cudaMemcpyAsync(d_pts, h_points, AB * (size_t)n, cudaMemcpyHostToDevice, st));
    } else {
        std::vector<char> packed(AB * (size_t)n);
        for (uint32_t k = 0; k < n; k++) memcpy(&packed[AB * k], h_points + AB * idx[k], AB);
        if (h_scalar_idx)
            for (uint32_t k = 0; k < n; k++) idx[k] = h_scalar_idx[idx[k]];
        ZKR_CUDA(cudaMemcpyAsync(d_pts, packed.data(), AB * (size_t)n, cudaMemcpyHostToDevice, st));
        ZKR_CUDA(cudaStreamSynchronize(st));
        ZKR_CUDA(cudaMalloc(&b->src_index, 4 * (size_t)n));
        ZKR_CUDA(cudaMemcpyAsync(b->src_index, idx.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, st));
        ZKR_CUDA(cudaStreamSynchronize(st));
        b->bytes += 4 * (size_t)n;
    }
    const size_t tbytes = AB * (size_t)n * W;
    ZKR_CUDA(cudaMalloc(&b->table, tbytes));
    b->bytes += tbytes;
    ZKR_LAUNCH(ctx, (k_precompute<F>), ceil_div(n, 64), 64, 0, st, d_pts, b->table, n, b->plan.c, W);
    ZKR_CUDA(cudaStreamSynchronize(st));
    ZKR_CUDA(cudaFree(d_pts));

    // work buffers
    MsmWork& wk = b->work;
    const size_t total = (size_t)W * n;
    b->logL = total >= (1u << 22) ? 5 : (total >= (1u << 16) ? 4 : 3);
    const size_t L = (size_t)1 << b->logL;
    const size_t T1 = (total + L - 1) / L;
    b->T1p = (uint32_t)(((T1 + kAccumThreads - 1) / kAccumThreads) * kAccumThreads);
    for (int i = 0; i < 2; i++) {
        ZKR_CUDA(cudaMalloc(&wk.keys[i], 4 * total));
        ZKR_CUDA(cudaMalloc(&wk.vals[i], 4 * total));
        wk.bytes += 8 * total;
    }
    cub::DoubleBuffer<uint32_t> dk(wk.keys[0], wk.keys[1]), dv(wk.vals[0], wk.vals[1]);
    ZKR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, wk.cub_bytes, dk, dv, (int)total, 0, b->plan.c, st));
    ZKR_CUDA(cudaMalloc(&wk.cub_tmp, wk.cub_bytes ? wk.cub_bytes : 1));
    ZKR_CUDA(cudaMalloc(&wk.buckets, XB * (size_t)b->plan.nbuckets));
    const size_t bnd0 = 2 * (size_t)b->T1p;
    const size_t lvl = 2;                 // smallest per-thread count any boundary level may use (level_log >= 1)
    size_t bnd1 = 2 * (((bnd0 + lvl - 1) / lvl + 63) / 64 * 64);
    if (bnd1 < 2 * (size_t)kFinishThreads) bnd1 = 2 * (size_t)kFinishThreads;
    ZKR_CUDA(cudaMalloc(&wk.bnd[0], XB * bnd0));
    ZKR_CUDA(cudaMalloc(&wk.bnd[1], XB * bnd1));
    ZKR_CUDA(cudaMalloc(&wk.bnd_keys[0], 4 * bnd0));
    ZKR_CUDA(cudaMalloc(&wk.bnd_keys[1], 4 * bnd1));
    const int rlc = (b->plan.c - 1) / 2, rlr = b->plan.c - 1 - rlc;
    const size_t nred = ((size_t)1 << rlr) + ((size_t)1 << rlc) + 32;
    ZKR_CUDA(cudaMalloc(&wk.red, XB * nred));
    ZKR_CUDA(cudaMalloc(&wk.red_counter, sizeof(unsigned int)));
    ZKR_CUDA(cudaMemsetAsync(wk.red_counter, 0, sizeof(unsigned int), st));
    ZKR_CUDA(cudaMalloc(&wk.result, XB));
    ZKR_CUDA(cudaMalloc(&wk.run_lo, 8 * (size_t)b->plan.nbuckets));
    wk.run_hi = wk.run_lo + b->plan.nbuckets;
    wk.bytes += 8 * (size_t)b->plan.nbuckets;
    ZKR_CUDA(cudaMalloc(&wk.range_err, sizeof(int)));
    ZKR_CUDA(cudaMemsetAsync(wk.range_err, 0, sizeof(int), st));
    wk.bytes += wk.cub_bytes + XB * ((size_t)b->plan.nbuckets + bnd0 + bnd1 + nred + 1) + 4 * (bnd0 + bnd1);
    b->bytes += wk.bytes;
    // per device, so once per work-buffer allocation rather than once per process (cold path, idempotent): a process
    // that drives several GPUs must opt in to > 48 KB of dynamic shared memory on each of them
    ZKR_CUDA(cudaFuncSetAttribute((k_bucket_sums<F, kReduceThreads>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(XB * kReduceThreads)));
    ZKR_CUDA(cudaFuncSetAttribute((k_bucket_weighted<F, kReduceThreads>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(XB * kReduceThreads)));
    constexpr bool kPrefetch = sizeof(F) == 32;
    ZKR_CUDA(cudaFuncSetAttribute((k_accum_affine<F, kPrefetch, 0>), cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    ZKR_CUDA(cudaFuncSetAttribute((k_accum_affine<F, kPrefetch, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    if (sizeof(F) == 32)
        ZKR_CUDA(cudaFuncSetAttribute((k_accum_affine<F, kPrefetch, sizeof(F) == 32 ? 2 : 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    ZKR_CUDA(cudaFuncSetAttribute(k_bucket_gather<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(XB * kGatherThreads)));
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

// One sorted (bucket, table entry) list -> bucket sums: level-1 accumulation, then the gather or the boundary levels.
// nbk buckets, nbk is also the sentinel key; msm_run passes its base set's buffers, msm_run_many a batch's.
struct AccumView {
    const uint32_t *skeys, *svals;
    uint32_t total, nbk, T1p;
    int logL;
    void* buckets;
    void* const* bnd;
    uint32_t* const* bnd_keys;
    uint32_t* run_lo;
};

template <class F>
int accumulate(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, const AccumView& v) {
    constexpr size_t XB = 4 * sizeof(F);
    constexpr bool kPrefetch = sizeof(F) == 32;    // G2 is register-bound; no software prefetch there
    const int c = b->plan.c;
    const uint32_t nb = v.nbk, total = v.total;
    const uint32_t *skeys = v.skeys, *svals = v.svals;
    ZKR_CUDA(cudaMemsetAsync(v.buckets, 0, XB * (size_t)nb, st));

    // level 1
    const int L = 1 << v.logL;
    const size_t smem = (size_t)(kAccumThreads / 32) * 2 * 32 * (L + 1) * 4;
    XYZZ<F>* buckets = (XYZZ<F>*)v.buckets;
    const int pslot = ctx->prof_begin(sizeof(F) == 32 ? PROF_ACCUM_G1 : PROF_ACCUM_G2, st, (double)total);
    // Boundary partials -> buckets: the one-launch gather up to 20-bit windows (every proof size), the round-1 recursive
    // levels above: at 22-bit windows the 12-bit top window puts n / 4096 extra entries into each of the 4096 lowest buckets,
    // i.e. thousands of moderately heavy buckets, which the whole-CTA heavy path handles badly (2^24: 48 vs 40.6 ms,
    // profiles/r02_msm_gather_vs_levels.json).
    // ZKR_MSM_LEVELS = 0 / 1 forces the gather / the levels (A/B knob).
    static const int force_levels = getenv("ZKR_MSM_LEVELS") ? atoi(getenv("ZKR_MSM_LEVELS")) : -1;
    const bool use_levels = force_levels >= 0 ? force_levels != 0 : c > 20;
    if (!use_levels) ZKR_CUDA(cudaMemsetAsync(v.run_lo, 0xff, 4 * (size_t)nb, st));
    // ZKR_LAZY: bit 0 = G1, bit 1 = G2 use the lazily reduced mixed addition, bit 2 = G1 additionally squares with
    // mont_sqr_raw (A/B knob; bit-identical results)
    const char* lazy_env = getenv("ZKR_LAZY");             // read per call: the GPU tests flip it inside one process
    const int lazy_mask = lazy_env ? atoi(lazy_env) : kLazyDefault;
    const int variant = !(lazy_mask & (sizeof(F) == 32 ? 1 : 2)) ? 0 : (sizeof(F) == 32 && (lazy_mask & 4)) ? 2 : 1;
    auto launch = [&](auto kern) -> int {
        ZKR_LAUNCH(ctx, kern, v.T1p / kAccumThreads, kAccumThreads, smem, st, skeys, svals, total, v.logL, b->table, buckets,
                   (XYZZ<F>*)v.bnd[0], use_levels ? v.bnd_keys[0] : nullptr, nb, use_levels ? nullptr : v.run_lo);
        return ZKR_OK;
    };
    int lrc;
    if (variant == 2) lrc = launch(k_accum_affine<F, kPrefetch, sizeof(F) == 32 ? 2 : 1>);
    else if (variant == 1) lrc = launch(k_accum_affine<F, kPrefetch, 1>);
    else lrc = launch(k_accum_affine<F, kPrefetch, 0>);
    if (lrc != ZKR_OK) return lrc;
    ctx->prof_end(sizeof(F) == 32 ? PROF_ACCUM_G1 : PROF_ACCUM_G2, pslot, st);
    if (!use_levels) {
        ZKR_LAUNCH(ctx, k_bucket_gather<F>, kHeavyBlocks + ceil_div(nb, kGatherThreads), kGatherThreads, XB * kGatherThreads,
                   st, skeys, total, v.logL, v.run_lo, (const XYZZ<F>*)v.bnd[0], buckets, nb);
    }
    // boundary levels (round-1 path)
    size_t cnt = 2 * (size_t)v.T1p;
    int cur = 0;
    for (; use_levels;) {
        const int llog = level_log(cnt);
        const size_t lvl = (size_t)1 << llog;
        if (cnt <= kFinishMax) {
            ZKR_LAUNCH(ctx, k_accum_finish<F>, 1, kFinishThreads, 0, st, v.bnd_keys[cur], (XYZZ<F>*)v.bnd[cur],
                       v.bnd_keys[cur ^ 1], (XYZZ<F>*)v.bnd[cur ^ 1], (uint32_t)cnt, buckets, nb);
            break;
        }
        const bool fin = cnt <= lvl;
        const size_t T = (cnt + lvl - 1) / lvl;
        const unsigned blocks = (unsigned)((T + 63) / 64);
        ZKR_LAUNCH(ctx, k_accum_xyzz<F>, blocks, 64, 0, st, v.bnd_keys[cur], (const XYZZ<F>*)v.bnd[cur],
                   (uint32_t)cnt, llog, buckets, (XYZZ<F>*)v.bnd[cur ^ 1], v.bnd_keys[cur ^ 1], nb, fin);
        if (fin) break;
        cnt = 2 * T;          // threads past T only pad their block; their slots are never read
        cur ^= 1;
    }
    return ZKR_OK;
}

template <class F>
int msm_run(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, const uint32_t* d_scalars, XYZZ<F>* d_out,
            const MsmHooks* hooks) {
    constexpr size_t XB = 4 * sizeof(F);
    const uint32_t n = b->n;
    if (n == 0) {
        ZKR_CUDA(cudaMemsetAsync(d_out, 0, XB, st));
        return ZKR_OK;
    }
    const MsmWork& wk = b->work;
    const int c = b->plan.c, W = b->plan.W;
    const uint32_t nb = b->plan.nbuckets;
    const uint32_t total = (uint32_t)W * n;
    const uint32_t *skeys, *svals;
    if (hooks && hooks->sorted_from) {
        const zkr_bases* o = hooks->sorted_from;
        if (o->n != n || o->plan.c != c || o->map_hash != b->map_hash || !o->work.sorted_keys) {
            set_error("msm_run: the base sets do not share a sort (different point maps or window plans)");
            return ZKR_E_INVALID;
        }
        skeys = o->work.sorted_keys;
        svals = o->work.sorted_vals;
    } else {
        ZKR_LAUNCH(ctx, k_digits, ceil_div(n, 128), 128, 0, st, d_scalars, b->src_index, n, c, W, nb, wk.keys[0],
                   wk.vals[0], wk.range_err);
        cub::DoubleBuffer<uint32_t> dk(wk.keys[0], wk.keys[1]), dv(wk.vals[0], wk.vals[1]);
        size_t tmp = wk.cub_bytes;
        ZKR_CUDA(cub::DeviceRadixSort::SortPairs(wk.cub_tmp, tmp, dk, dv, (int)total, 0, c, st));
        ctx->launches += 4;   // CUB: histogram + onesweep passes (not this library's own kernels, counted as a block)
        skeys = wk.sorted_keys = dk.Current();
        svals = wk.sorted_vals = dv.Current();
        if (hooks && hooks->ev_sorted) ZKR_CUDA(cudaEventRecord(hooks->ev_sorted, st));
    }
    const AccumView v = {skeys, svals, total, nb, b->T1p, b->logL, wk.buckets, wk.bnd, wk.bnd_keys, wk.run_lo};
    ZKR_TRY(accumulate<F>(ctx, st, b, v));
    // bucket reduction: row / column sums, then bit-decomposed weighted sums (see k_bucket_sums)
    const int lc = (c - 1) / 2, lr = c - 1 - lc;
    ZKR_LAUNCH(ctx, (k_bucket_sums<F, kReduceThreads>), (1u << lr) + (1u << lc), kReduceThreads, XB * kReduceThreads, st,
               (const XYZZ<F>*)wk.buckets, lr, lc, (XYZZ<F>*)wk.red);
    ZKR_LAUNCH(ctx, (k_bucket_weighted<F, kReduceThreads>), lr + lc + 1, kReduceThreads, XB * kReduceThreads, st, (XYZZ<F>*)wk.red, lr, lc,
               wk.red_counter, d_out);
    return ZKR_OK;
}

// ------------------------------------------------------------------------------------------------ batched MSM
// Sort keys of a batch of k vectors: k * nbuckets + 1 values (the zero-digit sentinel is k * nbuckets).
inline int many_key_bits(int c, int k) {
    int lg = 0;
    while ((1 << lg) < k) lg++;
    return c - 1 + lg + 1;
}

// ZKR_E_UNSUPPORTED, with the limit named, when k vectors over b do not fit one sort.
inline int many_limits(const zkr_bases* b, int k) {
    if (k < 1 || k > kMaxBatch) {
        set_error("batch of %d vectors: 1 .. %d per call", k, kMaxBatch);
        return k < 1 ? ZKR_E_INVALID : ZKR_E_UNSUPPORTED;
    }
    const uint64_t entries = (uint64_t)k * b->plan.W * b->n;
    if (entries >= (1ull << 31)) {
        set_error("batch of %d vectors: %d x %d windows x %u points = %llu sort entries, the limit is < 2^31", k, k,
                  b->plan.W, b->n, (unsigned long long)entries);
        return ZKR_E_UNSUPPORTED;
    }
    if (many_key_bits(b->plan.c, k) > 31) {
        set_error("batch of %d vectors: sort keys of %d bits at %d-bit windows, the limit is 31 bits", k,
                  many_key_bits(b->plan.c, k), b->plan.c);
        return ZKR_E_UNSUPPORTED;
    }
    return ZKR_OK;
}

template <class F>
int many_alloc(const zkr_bases* b, int cap, bool sorts, cudaStream_t st, MsmMany* w) {
    constexpr size_t XB = 4 * sizeof(F);
    ZKR_TRY(many_limits(b, cap));
    w->cap = cap;
    const uint32_t n = b->n;
    if (n == 0) return ZKR_OK;
    const int c = b->plan.c;
    const size_t nbk = (size_t)cap * b->plan.nbuckets;
    const size_t total = (size_t)cap * b->plan.W * n;
    auto dmalloc = [&](auto** p, size_t bytes) -> int {
        ZKR_CUDA(cudaMalloc(p, bytes ? bytes : 1));
        w->bytes += bytes;
        return ZKR_OK;
    };
    // as bases_build, for the batch's entry count
    w->logL = total >= (1u << 22) ? 5 : (total >= (1u << 16) ? 4 : 3);
    const size_t L = (size_t)1 << w->logL;
    const size_t T1 = (total + L - 1) / L;
    w->T1p = (uint32_t)(((T1 + kAccumThreads - 1) / kAccumThreads) * kAccumThreads);
    if (sorts) {
        for (int i = 0; i < 2; i++) {
            ZKR_TRY(dmalloc(&w->keys[i], 4 * total));
            ZKR_TRY(dmalloc(&w->vals[i], 4 * total));
        }
        cub::DoubleBuffer<uint32_t> dk(w->keys[0], w->keys[1]), dv(w->vals[0], w->vals[1]);
        ZKR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, w->cub_bytes, dk, dv, (int)total, 0, many_key_bits(c, cap), st));
        ZKR_TRY(dmalloc(&w->cub_tmp, w->cub_bytes));
    }
    ZKR_TRY(dmalloc(&w->buckets, XB * nbk));
    const size_t bnd0 = 2 * (size_t)w->T1p;
    size_t bnd1 = 2 * (((bnd0 + 1) / 2 + 63) / 64 * 64);
    if (bnd1 < 2 * (size_t)kFinishThreads) bnd1 = 2 * (size_t)kFinishThreads;
    ZKR_TRY(dmalloc(&w->bnd[0], XB * bnd0));
    ZKR_TRY(dmalloc(&w->bnd[1], XB * bnd1));
    ZKR_TRY(dmalloc(&w->bnd_keys[0], 4 * bnd0));
    ZKR_TRY(dmalloc(&w->bnd_keys[1], 4 * bnd1));
    const int rlc = (c - 1) / 2, rlr = c - 1 - rlc;
    w->nred = (1u << rlr) + (1u << rlc) + 32;
    ZKR_TRY(dmalloc(&w->red, XB * w->nred * (size_t)cap));
    ZKR_TRY(dmalloc(&w->red_counter, sizeof(unsigned int) * cap));
    ZKR_CUDA(cudaMemsetAsync(w->red_counter, 0, sizeof(unsigned int) * cap, st));
    ZKR_TRY(dmalloc(&w->run_lo, 8 * nbk));
    ZKR_TRY(dmalloc(&w->range_err, sizeof(int) * cap));
    ZKR_CUDA(cudaMemsetAsync(w->range_err, 0, sizeof(int) * cap, st));
    ZKR_TRY(dmalloc(&w->result, XB * cap));
    ZKR_CUDA(cudaFuncSetAttribute((k_bucket_sums_many<F, kReduceThreads>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(XB * kReduceThreads)));
    ZKR_CUDA(cudaFuncSetAttribute((k_bucket_weighted_many<F, kReduceThreads>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(XB * kReduceThreads)));
    ZKR_CUDA(cudaStreamSynchronize(st));
    return ZKR_OK;
}

template <class F>
int msm_run_many(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, MsmMany* w, int k, const uint32_t* d_scalars,
                 size_t stride, void* d_out, size_t out_stride, const MsmMany* sorted_from, cudaEvent_t ev_sorted) {
    constexpr size_t XB = 4 * sizeof(F);
    if (k < 1 || k > w->cap) {
        set_error("msm_run_many: %d vectors, the work buffers hold %d", k, w->cap);
        return ZKR_E_INVALID;
    }
    const uint32_t n = b->n;
    if (n == 0) {
        ZKR_CUDA(cudaMemset2DAsync(d_out, out_stride, 0, XB, k, st));
        return ZKR_OK;
    }
    const int c = b->plan.c, W = b->plan.W;
    const uint32_t nb = b->plan.nbuckets, nbk = nb * (uint32_t)k;
    const uint32_t total = (uint32_t)k * W * n;
    if (sorted_from) {
        if (!sorted_from->sorted_keys) {
            set_error("msm_run_many: the base set to share a sort with has not sorted this batch");
            return ZKR_E_INVALID;
        }
        w->sorted_keys = sorted_from->sorted_keys;
        w->sorted_vals = sorted_from->sorted_vals;
    } else {
        ZKR_LAUNCH(ctx, k_digits_many, dim3(ceil_div(n, 128), k), 128, 0, st, d_scalars, stride, b->src_index, n, c, W, nb,
                   nbk, w->keys[0], w->vals[0], w->range_err);
        cub::DoubleBuffer<uint32_t> dk(w->keys[0], w->keys[1]), dv(w->vals[0], w->vals[1]);
        const int bits = many_key_bits(c, k);
        size_t need = 0;
        ZKR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, dk, dv, (int)total, 0, bits, st));
        if (need > w->cub_bytes) {
            set_error("msm_run_many: the sort needs %zu bytes of scratch, %zu were sized", need, w->cub_bytes);
            return ZKR_E_INVALID;
        }
        ZKR_CUDA(cub::DeviceRadixSort::SortPairs(w->cub_tmp, need, dk, dv, (int)total, 0, bits, st));
        ctx->launches += 4;   // CUB, counted as a block (as msm_run)
        w->sorted_keys = dk.Current();
        w->sorted_vals = dv.Current();
        if (ev_sorted) ZKR_CUDA(cudaEventRecord(ev_sorted, st));
    }
    const AccumView v = {w->sorted_keys, w->sorted_vals, total, nbk, w->T1p, w->logL, w->buckets, w->bnd, w->bnd_keys, w->run_lo};
    ZKR_TRY(accumulate<F>(ctx, st, b, v));
    const int lc = (c - 1) / 2, lr = c - 1 - lc;
    ZKR_LAUNCH(ctx, (k_bucket_sums_many<F, kReduceThreads>), dim3((1u << lr) + (1u << lc), k), kReduceThreads, XB * kReduceThreads,
               st, (const XYZZ<F>*)w->buckets, nb, lr, lc, (XYZZ<F>*)w->red, w->nred);
    ZKR_LAUNCH(ctx, (k_bucket_weighted_many<F, kReduceThreads>), dim3(lr + lc + 1, k), kReduceThreads, XB * kReduceThreads, st,
               (XYZZ<F>*)w->red, w->nred, lr, lc, w->red_counter, (char*)d_out, out_stride);
    return ZKR_OK;
}

}  // namespace zkr
