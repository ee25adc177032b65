// Shared view of the NTT engine (ntt.cu) for the prover and the synthetic setup.
#pragma once
#include "common.cuh"
#include "fp.cuh"

namespace zkr {

struct NttRoots {
    Fr w, wi;        // omega_N, omega_N^-1
    Fr g, gi;        // omega_2N (coset shift), inverse
    Fr ninv;         // 1/N
    Fr hconst;       // R/(2N): mont_mul(x/R, .) = x/(2N)   (H pipeline final scaling)
    Fr one;
};

// Peer addressing of a sharded (multi-GPU) transform; all zero for a single GPU.
//   N = 2^n = 2^k0 rows x 2^s0 columns, G = 2^g ranks.
//   COLS slab of rank p: every row, columns [p C/G, (p+1) C/G): local[i * C/G + jl]   (natural-order data)
//   ROWS slab of rank q: rows [q R/G, (q+1) R/G), every column = a contiguous slice  (bit-reversed-order data)
constexpr int kMaxRanks = 8;
struct NttXchg {
    Fr* peer[kMaxRanks];
    int g, s0, k0, rank;
};

struct NttTables {
    int log_n = 0, kw = 0, lb = 0;
    NttRoots* roots = nullptr;
    Fr *wsub_f = nullptr, *wsub_i = nullptr;                              // omega_{2^kw}^{+-j}, j < 2^(kw-1)
    Fr *tw_lo_f = nullptr, *tw_hi_f = nullptr, *tw_lo_i = nullptr, *tw_hi_i = nullptr;  // omega_N^{+-X}
    Fr *cs_lo = nullptr, *cs_hi = nullptr, *cs_hi_n = nullptr;            // g^j ; hi / hi * 1/N
    Fr *ci_lo = nullptr, *ci_hi_n = nullptr, *ci_hi_h = nullptr;          // g^-j ; hi * 1/N ; hi * R/(2N)
    // Full-size tables, built on first use (ntt.cu): one modmul and one coalesced 32-byte read per element instead of
    // the two modmuls of a two-level lookup.  twfull_x[i]: inter-pass twiddles omega^(col * rev(row)) of pass i (laid out
    // like one chunk of that pass's data); cs_br / hf_br: the H pipeline's g^j / N and g^-j R/(2N) at j = bitrev(position).
    Fr *twfull_f[4] = {nullptr, nullptr, nullptr, nullptr}, *twfull_i[4] = {nullptr, nullptr, nullptr, nullptr};
    Fr *cs_br = nullptr, *hf_br = nullptr;
    size_t bytes = 0;
};

int ntt_get_tables(zkr_ctx* ctx, int log_n, NttTables** out);
// in-place; dit == false: natural in -> bit-reversed out (DIF); dit == true: bit-reversed in -> natural out
int ntt_run(zkr_ctx* ctx, cudaStream_t st, Fr* data, int log_n, bool dit, bool inverse);
// Sharded transform over the ranks of `x` (x.peer[r] = rank r's destination buffer, x.peer[x.rank] = dst).
//   dit == false: src = COLS slab, natural order  -> dst (on every rank) = ROWS slab, bit-reversed order
//   dit == true : src = ROWS slab, bit-reversed   -> dst = COLS slab, natural order  (src is clobbered)
// `barrier` is called twice on `st`: before the first remote store and after the last one.
int ntt_sharded_k0(int log_n, int g);
int ntt_run_sharded(zkr_ctx* ctx, cudaStream_t st, Fr* src, const NttXchg& x, int log_n, bool dit, bool inverse,
                    int (*barrier)(void*, cudaStream_t), void* barrier_arg);
// x[local] *= lo[j & mask] * hi[j >> lb] with j = the transform index of local element `local` of a slab
// (layout 0 = COLS / natural, 1 = ROWS / bit-reversed)
int ntt_scale_pow_sharded(zkr_ctx* ctx, cudaStream_t st, Fr* x, const NttXchg& g, int log_n, int layout,
                          const Fr* lo, const Fr* hi, int lb);
int ntt_scale_const(zkr_ctx* ctx, cudaStream_t st, Fr* x, size_t n, const Fr* cst);
int h_pipeline(zkr_ctx* ctx, cudaStream_t st, Fr* A, Fr* B, Fr* S, Fr* h, int log_m, bool bitrev_out);
// k pipelines in the launches of one: A, B, S, h each hold k vectors of 2^log_m elements back to back; h comes out in
// bit-reversed order per vector.  The 2 k transforms of A and B share one grid's y dimension.
int h_pipeline_many(zkr_ctx* ctx, cudaStream_t st, Fr* A, Fr* B, Fr* S, Fr* h, int log_m, int k);

}  // namespace zkr
