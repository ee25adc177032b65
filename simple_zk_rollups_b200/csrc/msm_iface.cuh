// Non-template view of the MSM engine for translation units that do not include msm.cuh
// (msm_api.cu, prover.cu): keeps them cheap to compile.  Implemented in msm_g1.cu / msm_g2.cu.
#pragma once
#include "common.cuh"

struct zkr_bases;
namespace zkr {
zkr_bases* bases_alloc();
int bases_group(const zkr_bases* b);
zkr_ctx* bases_ctx(const zkr_bases* b);
void bases_set_group(zkr_bases* b, int g);
int bases_build_g1(zkr_ctx*, zkr_bases*, const char* h_points, size_t n, int c_forced, cudaStream_t,
                   const uint32_t* h_scalar_idx);
int bases_build_g2(zkr_ctx*, zkr_bases*, const char* h_points, size_t n, int c_forced, cudaStream_t,
                   const uint32_t* h_scalar_idx);
// d_out: XYZZ point (128 B for G1, 256 B for G2), Montgomery
// Optional hooks (prover.cu): sorted_from = another base set whose sorted (bucket, point) pairs of THIS proof are
// consumed instead of extracting digits and sorting again (bases_share_sort must hold, and the stream must already
// wait for that set's ev_sorted); ev_sorted is recorded on the stream once the sorted pairs are final.
int msm_run_g1(zkr_ctx*, cudaStream_t, const zkr_bases*, const uint32_t* d_scalars, void* d_out,
               const zkr_bases* sorted_from = nullptr, cudaEvent_t ev_sorted = nullptr);
int msm_run_g2(zkr_ctx*, cudaStream_t, const zkr_bases*, const uint32_t* d_scalars, void* d_out,
               const zkr_bases* sorted_from = nullptr, cudaEvent_t ev_sorted = nullptr);
// same scalars, same compaction map, same window plan: one radix sort can serve both (B1' and B2' of a key)
bool bases_share_sort(const zkr_bases* a, const zkr_bases* b);
int g1_result_to_affine_std(zkr_ctx*, cudaStream_t, const void* d_xyzz, void* d_out64);
int g2_result_to_affine_std(zkr_ctx*, cudaStream_t, const void* d_xyzz, void* d_out128);
void bases_release(zkr_bases* b);
int bases_range_error(const zkr_bases* b, cudaStream_t st, int* err);
int bases_range_clear(const zkr_bases* b, cudaStream_t st);   // asynchronous, ordered on st
void bases_info(const zkr_bases* b, uint64_t* n, int* c, int* W, uint64_t* bytes);
void* bases_result_buf(const zkr_bases* b);
uint64_t bases_n_src(const zkr_bases* b);
int bases_peek(const zkr_bases* b, int what, size_t offset, void* out, size_t bytes);
}  // namespace zkr
