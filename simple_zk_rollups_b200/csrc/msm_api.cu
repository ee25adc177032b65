// C-ABI of the standalone MSM (zkr_bases_*, zkr_msm, zkr_msm_dev): the websnark g1_multiexp /
// g2_multiexp replacement exported for the sweeps of BASELINE.json configs[2].
#include "common.cuh"
#include "fp.cuh"

#include "msm_iface.cuh"
using namespace zkr;

extern "C" int zkr_bases_load(zkr_ctx* ctx, int group, const void* points, size_t n, int window_bits, zkr_bases** out) {
    if (!ctx || !out || (group != 1 && group != 2) || (!points && n) || window_bits < 0 || window_bits > 23 ||
        (window_bits > 0 && window_bits < 2))
        return ZKR_E_INVALID;
    *out = nullptr;
    DeviceGuard g(ctx->device);
    zkr_bases* b = bases_alloc();
    bases_set_group(b, group);
    int rc = group == 1 ? bases_build_g1(ctx, b, (const char*)points, n, window_bits, ctx->s[0], nullptr)
                        : bases_build_g2(ctx, b, (const char*)points, n, window_bits, ctx->s[0], nullptr);
    if (rc != ZKR_OK) {
        bases_release(b);
        return rc;
    }
    *out = b;
    return ZKR_OK;
}

extern "C" void zkr_bases_free(zkr_bases* b) {
    if (!b) return;
    DeviceGuard g(bases_ctx(b)->device);
    cudaDeviceSynchronize();
    bases_release(b);
}

extern "C" int zkr_bases_info(const zkr_bases* b, uint64_t* n_points, int* window_bits, int* n_windows, uint64_t* device_bytes) {
    if (!b) return ZKR_E_INVALID;
    bases_info(b, n_points, window_bits, n_windows, device_bytes);
    return ZKR_OK;
}

extern "C" int zkr_msm_dev(zkr_ctx* ctx, const zkr_bases* b, const void* d_scalars, size_t n, void* d_out_xyzz) {
    if (!ctx || !b || !d_scalars || !d_out_xyzz || bases_ctx(b) != ctx || n != bases_n_src(b)) {
        set_error("zkr_msm_dev: bad arguments (scalar count must equal the number of loaded points)");
        return ZKR_E_INVALID;
    }
    DeviceGuard g(ctx->device);
    return bases_group(b) == 1 ? msm_run_g1(ctx, ctx->user_stream, b, (const uint32_t*)d_scalars, d_out_xyzz)
                               : msm_run_g2(ctx, ctx->user_stream, b, (const uint32_t*)d_scalars, d_out_xyzz);
}

extern "C" int zkr_msm(zkr_ctx* ctx, const zkr_bases* b, const void* scalars, size_t n, int scalars_on_device, void* out_affine) {
    if (!ctx || !b || !scalars || !out_affine || bases_ctx(b) != ctx || n != bases_n_src(b)) {
        set_error("zkr_msm: bad arguments (scalar count must equal the number of loaded points)");
        return ZKR_E_INVALID;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->user_stream;
    const uint32_t* d_sc = (const uint32_t*)scalars;
    if (!scalars_on_device) {
        void* p;
        ZKR_TRY(ctx->scratch_get("msm_scalars", n * 32 + 32, &p));
        ZKR_CUDA(cudaMemcpyAsync(p, scalars, n * 32, cudaMemcpyHostToDevice, st));
        d_sc = (const uint32_t*)p;
    }
    const int group = bases_group(b);
    const size_t ob = group == 1 ? 64 : 128;
    void* res = bases_result_buf(b);
    void* d_aff;
    ZKR_TRY(ctx->scratch_get("msm_out", 256, &d_aff));
    if (n == 0 || res == nullptr) {
        memset(out_affine, 0, ob);
        return ZKR_OK;
    }
    if (group == 1) {
        ZKR_TRY(msm_run_g1(ctx, st, b, d_sc, res));
        ZKR_TRY(g1_result_to_affine_std(ctx, st, res, d_aff));
    } else {
        ZKR_TRY(msm_run_g2(ctx, st, b, d_sc, res));
        ZKR_TRY(g2_result_to_affine_std(ctx, st, res, d_aff));
    }
    ZKR_CUDA(cudaMemcpyAsync(out_affine, d_aff, ob, cudaMemcpyDeviceToHost, st));
    int err = 0;
    ZKR_TRY(bases_range_error(b, st, &err));
    ZKR_CUDA(cudaStreamSynchronize(st));
    if (err) {
        set_error("a scalar is >= r");
        return ZKR_E_WITNESS_RANGE;
    }
    return ZKR_OK;
}

extern "C" int zkr_msm_many(zkr_ctx* ctx, const zkr_bases* b, const void* scalars, size_t n, int n_vectors,
                            int scalars_on_device, void* out_affine) {
    if (!ctx || !b || !scalars || !out_affine || bases_ctx(b) != ctx || n != bases_n_src(b) || n_vectors < 1) {
        set_error("zkr_msm_many: bad arguments (n_vectors >= 1, scalar count per vector = the number of loaded points)");
        return ZKR_E_INVALID;
    }
    DeviceGuard g(ctx->device);
    cudaStream_t st = ctx->user_stream;
    const int group = bases_group(b);
    const size_t ob = group == 1 ? 64 : 128, xb = 2 * ob;
    const size_t k = (size_t)n_vectors;
    MsmMany* w;
    ZKR_TRY(bases_many_work(const_cast<zkr_bases*>(b), n_vectors, st, &w));
    if (bases_result_buf(b) == nullptr) {     // no finite point: every result is infinity
        memset(out_affine, 0, ob * k);
        return ZKR_OK;
    }
    const uint32_t* d_sc = (const uint32_t*)scalars;
    if (!scalars_on_device) {
        void* p;
        ZKR_TRY(ctx->scratch_get("msm_scalars", k * n * 32 + 32, &p));
        ZKR_CUDA(cudaMemcpyAsync(p, scalars, k * n * 32, cudaMemcpyHostToDevice, st));
        d_sc = (const uint32_t*)p;
    }
    void* d_aff;
    ZKR_TRY(ctx->scratch_get("msm_many_out", ob * k, &d_aff));
    void* res = msm_many_result_buf(w);
    ZKR_TRY(msm_many_run(ctx, st, b, w, n_vectors, d_sc, n, res, xb));
    ZKR_TRY(results_to_affine_std_many(ctx, st, group, res, n_vectors, d_aff));
    ZKR_CUDA(cudaMemcpyAsync(out_affine, d_aff, ob * k, cudaMemcpyDeviceToHost, st));
    int bad = -1;
    ZKR_TRY(msm_many_range_error(w, n_vectors, st, &bad));
    if (bad >= 0) {
        set_error("vector %d has a scalar >= r", bad);
        return ZKR_E_WITNESS_RANGE;
    }
    return ZKR_OK;
}

extern "C" int zkr_test_bases_peek(const zkr_bases* b, int what, size_t offset, void* out, size_t bytes) {
    if (!b || !out) return ZKR_E_INVALID;
    DeviceGuard g(bases_ctx(b)->device);
    return bases_peek(b, what, offset, out, bytes);
}
