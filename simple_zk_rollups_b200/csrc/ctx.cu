// libzkr context / error plumbing (C-ABI: zkr_ctx_*, zkr_strerror, zkr_last_error, zkr_version).
// zkr_ctx_create stands where the reference calls buildBn128()
// (/root/reference/operator/src/snarks/common.ts:23) -- but it is created once, not per proof.
#include "common.cuh"

namespace zkr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
    if (e == cudaErrorMemoryAllocation) return ZKR_E_NOMEM;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return ZKR_E_NO_DEVICE;
    return ZKR_E_CUDA;
}

void ntt_tables_free(NttTables* t);   // ntt.cu

}  // namespace zkr

using namespace zkr;

extern "C" const char* zkr_strerror(int code) {
    switch (code) {
        case ZKR_OK: return "ok";
        case ZKR_E_INVALID: return "invalid argument";
        case ZKR_E_BADKEY: return "malformed proving key";
        case ZKR_E_WITNESS_RANGE: return "witness value out of range";
        case ZKR_E_CUDA: return "CUDA error";
        case ZKR_E_NO_DEVICE: return "no usable CUDA device (this library has no CPU fallback)";
        case ZKR_E_NOMEM: return "out of device memory";
        case ZKR_E_NCCL: return "NCCL error";
        case ZKR_E_UNSUPPORTED: return "unsupported";
        default: return "unknown error";
    }
}

extern "C" const char* zkr_last_error(void) { return g_err; }

extern "C" const char* zkr_version(void) { return "zkr 0.1 (BN254 Groth16, sm_100a)"; }

extern "C" int zkr_ctx_create(int device, zkr_ctx** out) {
    if (!out) return ZKR_E_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("no CUDA device visible (%s); libzkr has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return ZKR_E_NO_DEVICE;
    }
    if (device < 0 || device >= count) {
        set_error("device %d out of range (0..%d)", device, count - 1);
        return ZKR_E_INVALID;
    }
    cudaDeviceProp prop;
    ZKR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this build only carries sm_100a code", device, prop.major, prop.minor);
        return ZKR_E_NO_DEVICE;
    }
    DeviceGuard g(device);
    // Out-of-line G2 helpers nest 256-byte by-value frames; give every thread a generous stack.
    ZKR_CUDA(cudaDeviceSetLimit(cudaLimitStackSize, 16 * 1024));
    zkr_ctx* c = new zkr_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    // Equal (default) stream priorities on purpose.  Round 1 (profiles/r01_sched_sweep.json, 2^20, real blinding
    // scalars): nine priority assignments over the five chains land within 17.12 .. 17.63 ms of the 17.22 ms of equal
    // priorities (H + A + B1 high: 18.3 ms); two and three proofs in flight per GPU gain 3 % in proofs/s
    // (profiles/r01_pipeline_check.json).  Round 2 (profiles/r02_schedule_ab.json, r02_priority_hsplit_ab.json): no
    // assignment is faster with two proofs in flight, as the throughput API runs.  The GPU is saturated by the proof's
    // bulk kernels; ordering them does not change the total.  (A first sweep with r = s = 0 favoured "B2 highest": with
    // zero scalars the two blinding multiplications are free, which hides that they then end up on the critical path.)
    for (int i = 0; i < kNumStreams; i++) {
        ZKR_CUDA(cudaStreamCreateWithFlags(&c->s[i], cudaStreamNonBlocking));
        ZKR_CUDA(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
    }
    ZKR_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    *out = c;
    return ZKR_OK;
}

extern "C" void zkr_ctx_destroy(zkr_ctx* c) {
    if (!c) return;
    DeviceGuard g(c->device);
    cudaDeviceSynchronize();
    for (auto& kv : c->ntt) ntt_tables_free(kv.second);
    for (auto& kv : c->scratch) cudaFree(kv.second.p);
    for (int i = 0; i < kNumStreams; i++) {
        cudaStreamDestroy(c->s[i]);
        cudaEventDestroy(c->ev_join[i]);
    }
    cudaEventDestroy(c->ev_fork);
    for (auto& r : c->prof)
        for (auto& e : r.ev)
            if (e) cudaEventDestroy(e);
    delete c;
}

extern "C" int zkr_ctx_set_stream(zkr_ctx* c, void* stream) {
    if (!c) return ZKR_E_INVALID;
    c->user_stream = (cudaStream_t)stream;
    return ZKR_OK;
}

extern "C" int zkr_ctx_synchronize(zkr_ctx* c) {
    if (!c) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaStreamSynchronize(c->user_stream));
    for (int i = 0; i < kNumStreams; i++) ZKR_CUDA(cudaStreamSynchronize(c->s[i]));
    return ZKR_OK;
}

extern "C" uint64_t zkr_ctx_kernel_launches(const zkr_ctx* c) { return c ? c->launches : 0; }

int zkr_ctx::scratch_get(const char* name, size_t bytes, void** out) {
    DevBuf& b = scratch[name];
    if (b.cap < bytes) {
        if (b.p) {
            // the old buffer may still be in use by queued work
            ZKR_CUDA(cudaDeviceSynchronize());
            ZKR_CUDA(cudaFree(b.p));
            b.p = nullptr;
            b.cap = 0;
        }
        size_t cap = (bytes + 255) & ~size_t(255);
        ZKR_CUDA(cudaMalloc(&b.p, cap));
        b.cap = cap;
    }
    *out = b.p;
    return ZKR_OK;
}

int zkr_ctx::fork(int n) {
    ZKR_CUDA(cudaEventRecord(ev_fork, user_stream));
    for (int i = 0; i < n; i++) ZKR_CUDA(cudaStreamWaitEvent(s[i], ev_fork, 0));
    return ZKR_OK;
}

int zkr_ctx::join(int n) {
    for (int i = 0; i < n; i++) {
        ZKR_CUDA(cudaEventRecord(ev_join[i], s[i]));
        ZKR_CUDA(cudaStreamWaitEvent(user_stream, ev_join[i], 0));
    }
    return ZKR_OK;
}

extern "C" int zkr_dev_malloc(zkr_ctx* c, size_t bytes, void** d_out) {
    if (!c || !d_out) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaMalloc(d_out, bytes ? bytes : 1));
    return ZKR_OK;
}

extern "C" int zkr_dev_free(zkr_ctx* c, void* d_ptr) {
    if (!c) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaStreamSynchronize(c->user_stream));
    ZKR_CUDA(cudaFree(d_ptr));
    return ZKR_OK;
}

extern "C" int zkr_dev_upload(zkr_ctx* c, void* d_dst, const void* h_src, size_t bytes) {
    if (!c || !d_dst || !h_src) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->user_stream));
    ZKR_CUDA(cudaStreamSynchronize(c->user_stream));   // h_src may be pageable and short-lived
    return ZKR_OK;
}

extern "C" int zkr_dev_download(zkr_ctx* c, void* h_dst, const void* d_src, size_t bytes) {
    if (!c || !h_dst || !d_src) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->user_stream));
    ZKR_CUDA(cudaStreamSynchronize(c->user_stream));
    return ZKR_OK;
}

int zkr_ctx::prof_begin(int id, cudaStream_t st, double units) {
    if (!profiling) return -1;
    zkr::ProfRing& r = prof[id];
    if (r.n >= zkr::kProfRing) return -1;
    const int slot = r.n++;
    for (int k = 0; k < 2; k++)
        if (!r.ev[2 * slot + k]) cudaEventCreate(&r.ev[2 * slot + k]);
    r.units += units;
    cudaEventRecord(r.ev[2 * slot], st);
    return slot;
}

void zkr_ctx::prof_end(int id, int slot, cudaStream_t st) {
    if (slot >= 0) cudaEventRecord(prof[id].ev[2 * slot + 1], st);
}

extern "C" int zkr_ctx_set_profile(zkr_ctx* c, int on) {
    if (!c) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaDeviceSynchronize());
    c->profiling = on != 0;
    for (auto& r : c->prof) {
        r.n = 0;
        r.units = 0;
    }
    return ZKR_OK;
}

extern "C" int zkr_ctx_set_serial(zkr_ctx* c, int on) {
    if (!c) return ZKR_E_INVALID;
    c->serial = on != 0;
    return ZKR_OK;
}

extern "C" int zkr_ctx_profile_read(zkr_ctx* c, int id, double* total_ms, int* launches, double* units) {
    if (!c || id < 0 || id >= PROF_COUNT) return ZKR_E_INVALID;
    DeviceGuard g(c->device);
    ZKR_CUDA(cudaDeviceSynchronize());
    ProfRing& r = c->prof[id];
    double tot = 0;
    for (int i = 0; i < r.n; i++) {
        float ms = 0;
        ZKR_CUDA(cudaEventElapsedTime(&ms, r.ev[2 * i], r.ev[2 * i + 1]));
        tot += ms;
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = r.n;
    if (units) *units = r.units;
    return ZKR_OK;
}
