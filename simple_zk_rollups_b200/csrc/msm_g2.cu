// G2 (Fq2 coordinates) instantiation of the MSM templates (msm.cuh).
#include "msm.cuh"
namespace zkr {
template int bases_build<Fq2>(zkr_ctx*, zkr_bases*, const char*, size_t, int, cudaStream_t, const uint32_t*);
template int msm_run<Fq2>(zkr_ctx*, cudaStream_t, const zkr_bases*, const uint32_t*, XYZZ<Fq2>*, const MsmHooks*);
int g2_result_to_affine_std(zkr_ctx* ctx, cudaStream_t st, const void* d_xyzz, void* d_out128) {
    ZKR_LAUNCH(ctx, k_xyzz_to_affine_std<Fq2>, 1, 1, 0, st, (const XYZZ<Fq2>*)d_xyzz, (char*)d_out128);
    return ZKR_OK;
}
}  // namespace zkr

namespace zkr {
int bases_build_g2(zkr_ctx* ctx, zkr_bases* b, const char* p, size_t n, int c, cudaStream_t st, const uint32_t* sidx) {
    b->ctx = ctx;
    return bases_build<Fq2>(ctx, b, p, n, c, st, sidx);
}
int msm_run_g2(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, const uint32_t* sc, void* out, const zkr_bases* sorted_from,
               cudaEvent_t ev_sorted) {
    MsmHooks h;
    h.sorted_from = sorted_from;
    h.ev_sorted = ev_sorted;
    return msm_run<Fq2>(ctx, st, b, sc, (XYZZ<Fq2>*)out, &h);
}
}  // namespace zkr
