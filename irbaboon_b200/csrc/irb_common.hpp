// irb_common.hpp -- host-side helpers shared by the translation units of libirb_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstddef>

#include "../../include/irb_b200.h"

namespace irbh {

int fail(int code, const char* fmt, ...);                      // records the thread's last error, returns code
int current_device();                                          // device chosen by irb_set_device on this thread
int twiddles(int dev, int M, const float2** out);              // table of the 2M roots exp(-2 pi i k / 2M), cached per (device, M)
// two-level table of the M-th roots: exp(-2 pi i idx / M) = hi[idx >> 10] * lo[idx & 1023], cached per (device, M)
int twiddles2(int dev, int M, const float2** hi, const float2** lo);
extern std::atomic<long long> g_launches;
extern thread_local int g_device;

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return irbh::fail(IRB_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Scratch memory of the offline functions is recycled through a small process-wide pool (blocks tagged with their device):
// cudaMalloc / cudaFree of the gigabytes a batched deconvolution needs cost tens to hundreds of milliseconds and vary from
// call to call.  irb_release_workspace() returns everything to the driver.  Engines never use the pool.
void* pool_get(int dev, size_t bytes, size_t* got);
void pool_put(int dev, void* p, size_t bytes);
size_t pool_release();

struct DevBuf {
    void* p = nullptr;
    size_t pooled_bytes = 0;       // > 0: the block goes back to the pool instead of cudaFree
    int pooled_dev = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) { if (pooled_bytes) pool_put(pooled_dev, p, pooled_bytes); else cudaFree(p); } }
    int alloc_scratch(size_t bytes, bool zero) {
        int dev = 0;
        CK(cudaGetDevice(&dev));
        const size_t want = bytes ? bytes : 16;
        p = pool_get(dev, want, &pooled_bytes);
        pooled_dev = dev;
        if (!p) {
            CK(cudaMalloc(&p, want));
            pooled_bytes = want;
        }
        if (zero) {
            CK(cudaMemset(p, 0, want));
            CK(cudaStreamSynchronize(cudaStreamLegacy));
        }
        return 0;
    }
    int alloc(size_t bytes, bool zero) {
        CK(cudaMalloc(&p, bytes ? bytes : 16));
        if (zero) {
            // cudaMemset runs on the legacy stream, asynchronously to the host, and the library's own streams are
            // non-blocking: wait for it here or a later copy on another stream could be overwritten by the zeros
            CK(cudaMemset(p, 0, bytes ? bytes : 16));
            CK(cudaStreamSynchronize(cudaStreamLegacy));
        }
        return 0;
    }
    template <typename T> T* as() const { return (T*) p; }
};

// device time of the kernels of this thread's most recent offline call (irb_last_compute_ms)
void set_last_compute_ms(double ms);

// brackets the kernel section(s) of an offline call with CUDA events and accumulates their elapsed time
struct ComputeTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st = nullptr;
    double total = 0.0;
    bool open = false;
    ~ComputeTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    int init(cudaStream_t s) { st = s; CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b)); return 0; }
    int begin() { CK(cudaEventRecord(a, st)); open = true; return 0; }
    int end() { CK(cudaEventRecord(b, st)); return 0; }
    int collect() {          // call after the stream was synchronised
        if (!open) return 0;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, a, b));
        total += ms; open = false;
        set_last_compute_ms(total);
        return 0;
    }
};

// DevBuf whose alloc() draws from the scratch pool: what the offline functions declare
struct ScratchBuf : DevBuf {
    int alloc(size_t bytes, bool zero) { return alloc_scratch(bytes, zero); }
};

// Declare a StreamGuard AFTER the scratch buffers its stream works on: destructors run in reverse order, so an early return
// first drains the stream (work already enqueued may still be reading or writing those buffers) and only then hands the
// buffers back to the process-wide pool, where another thread's call could pick them up.
struct StreamGuard {
    cudaStream_t s = nullptr;
    ~StreamGuard() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } }
    int create() { CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); return 0; }
};

inline int next_pow2(int x) {                                  // tools::nextPowerOfTwo, fp/tools.cpp:189-196
    if (x > 0 && (x & (x - 1)) == 0) return x;
    int r = 1;
    while (r <= x) r *= 2;
    return r;
}

}  // namespace irbh

struct irb_engine;
namespace irbh { int engine_mac_only(irb_engine* e, float* acc_dev); int engine_set_stamps(irb_engine* e, unsigned long long* dev); int engine_ir_copies(const irb_engine* e); }
