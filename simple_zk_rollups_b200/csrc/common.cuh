// Shared host-side plumbing of libzkr: context, error reporting, launch accounting.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <map>
#include <string>
#include <vector>

#include "../../include/zkr.h"

namespace zkr {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
// OS CSPRNG (getrandom), prover.cu: `bytes` random bytes / one scalar uniform in [0, r), 32 B std form
int os_random(void* out, size_t bytes);
int draw_scalar(void* out32);
// the scalar field modulus r, 8 x u32 little-endian (prover.cu)
extern const uint32_t kRModulus[8];

#define ZKR_CUDA(expr)                                                          \
    do {                                                                        \
        cudaError_t _e = (expr);                                                \
        if (_e != cudaSuccess) return zkr::cuda_fail(_e, #expr, __FILE__, __LINE__); \
    } while (0)

#define ZKR_TRY(expr)            \
    do {                         \
        int _rc = (expr);        \
        if (_rc != ZKR_OK) return _rc; \
    } while (0)

// Launch + count.  Every kernel of this library goes through here so that
// zkr_ctx_kernel_launches() / bench.py's "gpu_launches" is a count, not an estimate.
#define ZKR_LAUNCH(ctx, kern, grid, block, smem, stream, ...)                   \
    do {                                                                        \
        kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);               \
        (ctx)->launches++;                                                      \
        cudaError_t _e = cudaPeekAtLastError();                                 \
        if (_e != cudaSuccess) return zkr::cuda_fail(_e, #kern, __FILE__, __LINE__); \
    } while (0)

struct NttTables;   // ntt.cu
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

constexpr int kNumStreams = 6;      // s[0..4]: the proof's five chains, s[5]: witness uploads

// Per-kernel device timing for bench.py's roofline: rings of CUDA event pairs recorded on the
// launching stream around selected kernels while profiling is enabled.
enum ProfId { PROF_ACCUM_G1 = 0, PROF_ACCUM_G2 = 1, PROF_NTT_PASS = 2, PROF_NTT_XCHG = 3, PROF_COUNT = 4 };
constexpr int kProfRing = 512;
struct ProfRing {
    cudaEvent_t ev[2 * kProfRing] = {};
    int n = 0;
    double units = 0;     // caller-defined work units summed over the recorded launches
};

}  // namespace zkr

struct zkr_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t user_stream = nullptr;          // work is ordered after / before this stream
    cudaStream_t s[zkr::kNumStreams] = {};       // internal non-blocking streams
    cudaEvent_t ev_fork = nullptr;
    cudaEvent_t ev_join[zkr::kNumStreams] = {};
    uint64_t launches = 0;
    std::map<int, zkr::NttTables*> ntt;          // per log_n twiddle tables
    std::map<std::string, zkr::DevBuf> scratch;  // named, grow-only device scratch
    zkr_stats last_stats = {};
    bool profiling = false;
    bool serial = false;                         // run a proof's stages back to back on one stream
    zkr::ProfRing prof[zkr::PROF_COUNT];
    // returns the slot to pass to prof_end, or -1 when not recording
    int prof_begin(int id, cudaStream_t st, double units);
    void prof_end(int id, int slot, cudaStream_t st);

    // grow-only named scratch buffer on this ctx's device
    int scratch_get(const char* name, size_t bytes, void** out);
    int fork(int n);   // make streams s[0..n) wait for everything queued on user_stream
    int join(int n);   // make user_stream wait for s[0..n)
};

namespace zkr {

struct DeviceGuard {
    int prev = 0;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        cur = dev;
    }
    ~DeviceGuard() {
        if (prev != cur) cudaSetDevice(prev);
    }
    int cur;
};

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Device buffers of one call, freed when the call returns, on its error paths too.  A secret buffer is zeroed when it
// is allocated, and zeroed again on its stream before it is freed, so what it held never outlives the call.
struct DevAllocs {
    struct Buf {
        void* p;
        size_t wipe;            // bytes zeroed on `st` before the free; 0 for public buffers
        cudaStream_t st;
    };
    std::vector<Buf> bufs;

    DevAllocs() = default;
    DevAllocs(const DevAllocs&) = delete;
    DevAllocs& operator=(const DevAllocs&) = delete;
    ~DevAllocs() {
        for (const Buf& b : bufs)
            if (b.wipe) {
                cudaMemsetAsync(b.p, 0, b.wipe, b.st);
                cudaStreamSynchronize(b.st);
            }
        for (const Buf& b : bufs) cudaFree(b.p);
    }
    template <class T>
    int alloc(T** out, size_t bytes) {
        ZKR_CUDA(cudaMalloc(out, bytes ? bytes : 1));
        bufs.push_back({*out, 0, nullptr});
        return ZKR_OK;
    }
    template <class T>
    int alloc_secret(T** out, size_t bytes, cudaStream_t st) {
        ZKR_TRY(alloc(out, bytes));
        bufs.back().wipe = bytes;
        bufs.back().st = st;
        ZKR_CUDA(cudaMemsetAsync(*out, 0, bytes, st));
        return ZKR_OK;
    }
    // *d = a new buffer holding the `count` elements of T at host address h
    template <class T>
    int upload(T** d, const void* h, size_t count, cudaStream_t st) {
        ZKR_TRY(alloc(d, sizeof(T) * count));
        if (count) ZKR_CUDA(cudaMemcpyAsync(*d, h, sizeof(T) * count, cudaMemcpyHostToDevice, st));
        return ZKR_OK;
    }
    // frees a public buffer before the call returns
    void release(void* q) {
        for (size_t i = 0; i < bufs.size(); i++)
            if (bufs[i].p == q) {
                cudaFree(q);
                bufs.erase(bufs.begin() + i);
                return;
            }
    }
};

}  // namespace zkr
