// irb_benchaids.cu -- the bench-only translation unit of libirb_b200.so: everything declared in include/irb_b200_bench.h.
// Measurement aids and A/B switches live here, not in the product ABI (include/irb_b200.h) and not in the hot-path
// dispatch: the engine reads irbh::g_tuning (plain globals with compiled-in defaults); this file is their only writer.
#include <sys/mman.h>

#include <chrono>
#include <cstring>
#include <new>

#include "../../include/irb_b200_bench.h"
#include "irb_common.hpp"
#include "irb_kernels.cuh"
#include "irb_tuning.hpp"

namespace irb {
// read-only bandwidth probe (irbx_hbm_read_probe): every CTA walks the buffer grid-strided in 16 KB pieces, four independent
// 32-byte loads per thread in flight; the XOR of everything read is stored only if it equals a value it never takes
__device__ __forceinline__ void probe_store(float4* q, float4 v, int kind, uint64_t pol) {
    if (kind == 1) asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    else if (kind == 2) asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
    else if (kind == 3) asm volatile("st.global.wt.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    else if (kind == 4) asm volatile("st.global.cg.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(q), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    else *q = v;
}
static __global__ void __launch_bounds__(512) k_read_probe(float4* __restrict__ p, size_t n_pieces, unsigned* sink, int write_every, int store_kind) {
    uint64_t pol = 0;
    if (store_kind == 2) pol = l2_policy_evict_first();
    if (store_kind == 5) { asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol)); }
    const int sk = store_kind == 5 ? 2 : store_kind;
    unsigned acc = 0;
    size_t piece = blockIdx.x;
    for (; piece + 3 * (size_t) gridDim.x < n_pieces; piece += 4 * (size_t) gridDim.x) {
        float4 a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float4* q = p + (piece + u * (size_t) gridDim.x) * 1024 + 2 * threadIdx.x;         // 16 KB = 512 threads x 32 bytes
            const size_t pc = piece + u * (size_t) gridDim.x;
            if (write_every > 0 && pc % (size_t) write_every == 0) {                          // a share of the pieces is WRITTEN instead
                probe_store(q, make_float4(1.f, 2.f, 3.f, 4.f), sk, pol); probe_store(q + 1, make_float4(5.f, 6.f, 7.f, 8.f), sk, pol);
                a[u] = b[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            } else ldg_stream256(q, a[u], b[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) acc ^= __float_as_uint(a[u].x) ^ __float_as_uint(a[u].w) ^ __float_as_uint(b[u].y) ^ __float_as_uint(b[u].z);
    }
    for (; piece < n_pieces; piece += gridDim.x) {
        float4 a, b;
        ldg_stream256(p + piece * 1024 + 2 * threadIdx.x, a, b);
        acc ^= __float_as_uint(a.x) ^ __float_as_uint(a.w) ^ __float_as_uint(b.y) ^ __float_as_uint(b.z);
    }
    if (acc == 0x7fc12345u) *sink = acc;
}

}  // namespace irb

namespace {
using irbh::fail;
int* tuning_field(const char* name) {
    irbh::Tuning& t = irbh::g_tuning;
    struct { const char* n; int* p; } tab[] = {
        {"mac_persistent", &t.mac_persistent}, {"fuse_split", &t.fuse_split}, {"mac_tma", &t.mac_tma}, {"mac_wide", &t.mac_wide}, {"mac_u", &t.mac_u}, {"fdl_plain", &t.fdl_plain},
        {"producer_sleep_ns", &t.producer_sleep_ns}, {"no_graph", &t.no_graph}, {"deconv_sub", &t.deconv_sub}, {"deconv_streams", &t.deconv_streams}, {"avg_fused", &t.avg_fused}, {"deconv_groups", &t.deconv_groups}, {"deconv_group_cap", &t.deconv_group_cap}, {"release_fence", &t.release_fence}, {"release_dep", &t.release_dep},
        {"persistent_ctas", &t.persistent_ctas}, {"unit_narrowing", &t.unit_narrowing}, {"ir_replicas", &t.ir_replicas}, {"stagger_ns", &t.stagger_ns}, {"ring_stages", &t.ring_stages}};
    if (name) for (auto& e : tab) if (!strcmp(e.n, name)) return e.p;
    return nullptr;
}
}  // namespace

struct irbx_copy_probe {
    int device = 0, host_mode = 0;
    size_t bytes = 0, map_bytes = 0;
    float *h_in = nullptr, *h_out = nullptr, *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s_in = nullptr, s_out = nullptr;
};

extern "C" {

int irbx_set_tuning(const char* name, int value) {
    int* p = tuning_field(name);
    if (!p) return fail(IRB_ERR_ARG, "unknown tuning knob '%s'", name ? name : "(null)");
    *p = value;
    return 0;
}
int irbx_get_tuning(const char* name) {
    int* p = tuning_field(name);
    if (!p) return fail(IRB_ERR_ARG, "unknown tuning knob '%s'", name ? name : "(null)");
    return *p;
}

int irbx_engine_mac_only_device(irb_engine* e, float* acc_dev) { return irbh::engine_mac_only(e, acc_dev); }
int irbx_engine_set_stamps(irb_engine* e, unsigned long long* stamps_dev) { return irbh::engine_set_stamps(e, stamps_dev); }
int irbx_engine_ir_copies(const irb_engine* e) { return irbh::engine_ir_copies(e); }

int irbx_hbm_read_probe(size_t bytes, int iters, int write_every, int store_kind, double* gbs) {
    if (!gbs || iters < 1 || bytes < (1u << 20)) return fail(IRB_ERR_ARG, "bad argument");
    CK(cudaSetDevice(irbh::g_device));
    const size_t pieces = bytes / 16384;
    irbh::DevBuf buf, sink;
    int rc;
    if ((rc = buf.alloc(pieces * 16384, true)) || (rc = sink.alloc(sizeof(unsigned), true))) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, irbh::g_device);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int grid = sms * 4;                                  // 4 x 512 threads resident per SM
    irb::k_read_probe<<<grid, 512>>>(buf.as<float4>(), pieces, sink.as<unsigned>(), write_every, store_kind);
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) irb::k_read_probe<<<grid, 512>>>(buf.as<float4>(), pieces, sink.as<unsigned>(), write_every, store_kind);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaGetLastError());
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    irbh::g_launches += iters + 1;
    *gbs = (double) (pieces * 16384) * iters / (ms * 1e-3) / 1e9;
    return 0;
}

int irbx_copy_probe_destroy(irbx_copy_probe* p) {
    if (!p) return 0;
    cudaSetDevice(p->device);
    if (p->s_in) { cudaStreamSynchronize(p->s_in); cudaStreamDestroy(p->s_in); }
    if (p->s_out) { cudaStreamSynchronize(p->s_out); cudaStreamDestroy(p->s_out); }
    if (p->host_mode == 2) {
        if (p->h_in) { cudaHostUnregister(p->h_in); munmap(p->h_in, p->map_bytes); }
        if (p->h_out) { cudaHostUnregister(p->h_out); munmap(p->h_out, p->map_bytes); }
    } else {
        if (p->h_in) cudaFreeHost(p->h_in);
        if (p->h_out) cudaFreeHost(p->h_out);
    }
    if (p->d_in) cudaFree(p->d_in);
    if (p->d_out) cudaFree(p->d_out);
    cudaGetLastError();
    delete p;
    return 0;
}

int irbx_copy_probe_create(irbx_copy_probe** out, int device, size_t bytes, int host_mode) {
    if (!out || bytes < 4096 || host_mode < 0 || host_mode > 2) return fail(IRB_ERR_ARG, "bad argument");
    *out = nullptr;
    CK(cudaSetDevice(device));
    irbx_copy_probe* p = new (std::nothrow) irbx_copy_probe;
    if (!p) return fail(IRB_ERR_ARG, "out of host memory");
    p->device = device; p->host_mode = host_mode; p->bytes = bytes;
    cudaError_t ce = cudaSuccess;
    if (host_mode == 2) {
        const size_t huge = 2u << 20;
        p->map_bytes = (bytes + huge - 1) / huge * huge;
        void* a = mmap(nullptr, p->map_bytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        void* b = mmap(nullptr, p->map_bytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (a == MAP_FAILED || b == MAP_FAILED) { if (a != MAP_FAILED) munmap(a, p->map_bytes); if (b != MAP_FAILED) munmap(b, p->map_bytes); delete p; return fail(IRB_ERR_ARG, "mmap of %zu bytes failed", p->map_bytes); }
        madvise(a, p->map_bytes, MADV_HUGEPAGE); madvise(b, p->map_bytes, MADV_HUGEPAGE);
        memset(a, 1, p->map_bytes); memset(b, 0, p->map_bytes);                    // first touch: the pages exist before they are pinned
        p->h_in = (float*) a; p->h_out = (float*) b;
        ce = cudaHostRegister(a, p->map_bytes, cudaHostRegisterDefault);
        if (ce != cudaSuccess) { p->h_in = p->h_out = nullptr; munmap(a, p->map_bytes); munmap(b, p->map_bytes); }
        else if ((ce = cudaHostRegister(b, p->map_bytes, cudaHostRegisterDefault)) != cudaSuccess) { cudaHostUnregister(a); p->h_in = p->h_out = nullptr; munmap(a, p->map_bytes); munmap(b, p->map_bytes); }
    } else {
        ce = cudaHostAlloc((void**) &p->h_in, bytes, host_mode == 1 ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
        if (ce == cudaSuccess) ce = cudaHostAlloc((void**) &p->h_out, bytes, cudaHostAllocDefault);
        if (ce == cudaSuccess) { memset(p->h_in, 1, bytes); memset(p->h_out, 0, bytes); }
    }
    if (ce == cudaSuccess) ce = cudaMalloc((void**) &p->d_in, bytes);
    if (ce == cudaSuccess) ce = cudaMalloc((void**) &p->d_out, bytes);
    if (ce == cudaSuccess) ce = cudaMemset(p->d_out, 0, bytes);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) {
        const int rc = fail(IRB_ERR_CUDA, "copy probe setup: %s", cudaGetErrorString(ce));
        irbx_copy_probe_destroy(p);
        return rc;
    }
    *out = p;
    return 0;
}

int irbx_copy_probe_run(irbx_copy_probe* p, int iters, int direction, size_t chunk_bytes, double* seconds) {
    if (!p || !seconds || iters < 1 || direction < 1 || direction > 3) return fail(IRB_ERR_ARG, "bad argument");
    CK(cudaSetDevice(p->device));
    const size_t chunk = chunk_bytes ? (chunk_bytes + 15) / 16 * 16 : p->bytes;
    CK(cudaStreamSynchronize(p->s_in)); CK(cudaStreamSynchronize(p->s_out));
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < iters; ++i) {
        for (size_t off = 0; off < p->bytes; off += chunk) {
            const size_t n = off + chunk <= p->bytes ? chunk : p->bytes - off;
            if (direction & 1) CK(cudaMemcpyAsync((char*) p->d_in + off, (const char*) p->h_in + off, n, cudaMemcpyHostToDevice, p->s_in));
            if (direction & 2) CK(cudaMemcpyAsync((char*) p->h_out + off, (const char*) p->d_out + off, n, cudaMemcpyDeviceToHost, p->s_out));
        }
    }
    CK(cudaStreamSynchronize(p->s_in)); CK(cudaStreamSynchronize(p->s_out));
    *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return 0;
}

}  // extern "C"
