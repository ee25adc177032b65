// G1 instantiation of the MSM templates (msm.cuh).
#include "msm.cuh"
namespace zkr {
template int bases_build<Fq>(zkr_ctx*, zkr_bases*, const char*, size_t, int, cudaStream_t, const uint32_t*);
template int msm_run<Fq>(zkr_ctx*, cudaStream_t, const zkr_bases*, const uint32_t*, XYZZ<Fq>*, const MsmHooks*);
int g1_result_to_affine_std(zkr_ctx* ctx, cudaStream_t st, const void* d_xyzz, void* d_out64) {
    ZKR_LAUNCH(ctx, k_xyzz_to_affine_std<Fq>, 1, 1, 0, st, (const XYZZ<Fq>*)d_xyzz, (char*)d_out64);
    return ZKR_OK;
}
// G2 instantiations of the batched MSM (msm_g2.cu)
int many_alloc_g2(const zkr_bases* b, int cap, bool sorts, cudaStream_t st, MsmMany* w);
int msm_run_many_g2(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, MsmMany* w, int k, const uint32_t* sc, size_t stride,
                    void* out, size_t out_stride, const MsmMany* sorted_from, cudaEvent_t ev_sorted);
int g2_results_to_affine_std_many(zkr_ctx* ctx, cudaStream_t st, const void* d_xyzz, int k, void* d_out);

int msm_many_alloc(const zkr_bases* b, int cap, bool sorts, cudaStream_t st, MsmMany** out) {
    MsmMany* w = new MsmMany();
    const int rc = b->group == 1 ? many_alloc<Fq>(b, cap, sorts, st, w) : many_alloc_g2(b, cap, sorts, st, w);
    if (rc != ZKR_OK) {
        msm_many_free(w);
        return rc;
    }
    *out = w;
    return ZKR_OK;
}
void msm_many_free(MsmMany* w) {
    if (!w) return;
    void* ps[] = {w->keys[0], w->keys[1], w->vals[0], w->vals[1], w->cub_tmp, w->buckets, w->bnd[0], w->bnd[1],
                  w->bnd_keys[0], w->bnd_keys[1], w->red, w->red_counter, w->run_lo, w->range_err, w->result};
    for (void* p : ps) cudaFree(p);
    delete w;
}
uint64_t msm_many_bytes(const MsmMany* w) { return w ? w->bytes : 0; }
void* msm_many_result_buf(const MsmMany* w) { return w->result; }
int msm_many_run(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, MsmMany* w, int k, const uint32_t* sc, size_t stride,
                 void* out, size_t out_stride, const MsmMany* sorted_from, cudaEvent_t ev_sorted) {
    return b->group == 1 ? msm_run_many<Fq>(ctx, st, b, w, k, sc, stride, out, out_stride, sorted_from, ev_sorted)
                         : msm_run_many_g2(ctx, st, b, w, k, sc, stride, out, out_stride, sorted_from, ev_sorted);
}
int msm_many_range_error(const MsmMany* w, int k, cudaStream_t st, int* first_bad) {
    *first_bad = -1;
    if (!w->range_err) return ZKR_OK;
    std::vector<int> f(k);
    ZKR_CUDA(cudaMemcpyAsync(f.data(), w->range_err, sizeof(int) * k, cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    for (int j = 0; j < k && *first_bad < 0; j++)
        if (f[j]) *first_bad = j;
    if (*first_bad >= 0) ZKR_CUDA(cudaMemsetAsync(w->range_err, 0, sizeof(int) * k, st));
    return ZKR_OK;
}
int bases_many_work(zkr_bases* b, int k, cudaStream_t st, MsmMany** out) {
    if (!b->many || b->many->cap < k) {
        if (b->many) {
            ZKR_CUDA(cudaStreamSynchronize(st));
            b->bytes -= b->many->bytes;
            msm_many_free(b->many);
            b->many = nullptr;
        }
        ZKR_TRY(msm_many_alloc(b, k, true, st, &b->many));
        b->bytes += b->many->bytes;
    }
    *out = b->many;
    return ZKR_OK;
}
int results_to_affine_std_many(zkr_ctx* ctx, cudaStream_t st, int group, const void* d_xyzz, int k, void* d_out) {
    if (group != 1) return g2_results_to_affine_std_many(ctx, st, d_xyzz, k, d_out);
    ZKR_LAUNCH(ctx, k_xyzz_to_affine_std_many<Fq>, k, 1, 0, st, (const XYZZ<Fq>*)d_xyzz, (char*)d_out);
    return ZKR_OK;
}
}  // namespace zkr

// non-template glue used by msm_api.cu / prover.cu (they do not include msm.cuh)
namespace zkr {
zkr_bases* bases_alloc() { return new zkr_bases(); }
int bases_group(const zkr_bases* b) { return b->group; }
zkr_ctx* bases_ctx(const zkr_bases* b) { return b->ctx; }
void bases_set_group(zkr_bases* b, int g) { b->group = g; }
uint64_t bases_n_src(const zkr_bases* b) { return b->n_src; }
bool bases_share_sort(const zkr_bases* a, const zkr_bases* b) {
    return a && b && a->n && a->n == b->n && a->plan.c == b->plan.c && a->plan.W == b->plan.W && a->map_hash == b->map_hash;
}
void* bases_result_buf(const zkr_bases* b) { return b->work.result; }
void bases_info(const zkr_bases* b, uint64_t* n, int* c, int* W, uint64_t* bytes) {
    if (n) *n = b->n;
    if (c) *c = b->plan.c;
    if (W) *W = b->plan.W;
    if (bytes) *bytes = b->bytes;
}
int bases_build_g1(zkr_ctx* ctx, zkr_bases* b, const char* p, size_t n, int c, cudaStream_t st, const uint32_t* sidx) {
    b->ctx = ctx;
    return bases_build<Fq>(ctx, b, p, n, c, st, sidx);
}
int msm_run_g1(zkr_ctx* ctx, cudaStream_t st, const zkr_bases* b, const uint32_t* sc, void* out, const zkr_bases* sorted_from,
               cudaEvent_t ev_sorted) {
    MsmHooks h;
    h.sorted_from = sorted_from;
    h.ev_sorted = ev_sorted;
    return msm_run<Fq>(ctx, st, b, sc, (XYZZ<Fq>*)out, &h);
}
int bases_range_error(const zkr_bases* b, cudaStream_t st, int* err) {
    *err = 0;
    if (!b->work.range_err) return ZKR_OK;
    ZKR_CUDA(cudaMemcpyAsync(err, b->work.range_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    ZKR_CUDA(cudaStreamSynchronize(st));
    if (*err) ZKR_CUDA(cudaMemsetAsync(b->work.range_err, 0, sizeof(int), st));
    return ZKR_OK;
}
int bases_range_clear(const zkr_bases* b, cudaStream_t st) {
    if (b && b->work.range_err) ZKR_CUDA(cudaMemsetAsync(b->work.range_err, 0, sizeof(int), st));
    return ZKR_OK;
}
// white-box test hook: copy an internal device buffer to the host
int bases_peek(const zkr_bases* b, int what, size_t offset, void* out, size_t bytes) {
    const MsmWork& w = b->work;
    const void* src = nullptr;
    switch (what) {
        case 0: src = b->table; break;
        case 1: src = w.keys[0]; break;
        case 2: src = w.keys[1]; break;
        case 3: src = w.vals[0]; break;
        case 4: src = w.vals[1]; break;
        case 5: src = w.buckets; break;
        case 6: src = w.result; break;
        case 7: src = w.red; break;
        case 8: src = w.bnd_keys[0]; break;
        case 9: src = w.bnd_keys[1]; break;
        case 10: src = w.bnd[0]; break;
        case 11: src = w.bnd[1]; break;
        default: return ZKR_E_INVALID;
    }
    if (!src) return ZKR_E_INVALID;
    ZKR_CUDA(cudaDeviceSynchronize());
    ZKR_CUDA(cudaMemcpy(out, (const char*)src + offset, bytes, cudaMemcpyDeviceToHost));
    return ZKR_OK;
}
void bases_release(zkr_bases* b) {
    if (!b) return;
    MsmWork& w = b->work;
    void* ps[] = {b->src_index, b->table, w.keys[0], w.keys[1], w.vals[0], w.vals[1], w.cub_tmp, w.buckets,
                  w.bnd[0], w.bnd[1], w.bnd_keys[0], w.bnd_keys[1], w.red, w.red_counter, w.result, w.range_err,
                  w.run_lo};
    for (void* p : ps) cudaFree(p);
    msm_many_free(b->many);
    delete b;
}
}  // namespace zkr
