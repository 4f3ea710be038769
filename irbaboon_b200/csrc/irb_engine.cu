// irb_engine.cu -- host side of libirb_b200.so: the C ABI declared in include/irb_b200.h over the
// kernels in irb_kernels.cuh.  No CPU compute path exists in this file: every entry point either
// launches sm_100a kernels or fails with IRB_ERR_CUDA.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <new>
#include <vector>
#include <atomic>

#include "irb_common.hpp"
#include "irb_kernels.cuh"
#include "irb_ir_load.cuh"
#include "irb_mac_p.cuh"
#include "irb_mac_mx.cuh"
#include "irb_tuning.hpp"

namespace irbh {

Tuning g_tuning;

thread_local char g_err[512] = "";
thread_local int g_device = 0;
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int current_device() { return g_device; }
thread_local double g_last_compute_ms = 0.0;
void set_last_compute_ms(double ms) { g_last_compute_ms = ms; }

// FFT tables (irb_fft.cuh: fft_build_table), one per (device, M), built in double like the reference FFT's tables
int twiddles(int dev, int M, const float2** out) {
    struct Entry { int dev, M; float2* d; };
    static std::mutex mu;
    static std::vector<Entry> tab;
    std::lock_guard<std::mutex> lk(mu);
    for (auto& e : tab) if (e.dev == dev && e.M == M) { *out = e.d; return 0; }
    std::vector<float2> h((size_t) irb::fft_table_size(M));
    irb::fft_build_table(M, h.data());          // the N roots, then the per-thread twiddles of every pass (irb_fft.cuh)
    float2* d = nullptr;
    CK(cudaMalloc(&d, sizeof(float2) * h.size()));
    CK(cudaMemcpy(d, h.data(), sizeof(float2) * h.size(), cudaMemcpyHostToDevice));
    tab.push_back({dev, M, d});
    *out = d;
    return 0;
}

// ---- scratch pool ------------------------------------------------------------------------------------
namespace {
struct PoolBlock { void* p; size_t bytes; int dev; };
std::mutex g_pool_mu;
std::vector<PoolBlock> g_pool;
size_t g_pool_bytes = 0;
constexpr size_t kPoolCap = 12ull << 30;         // free blocks kept at most
}  // namespace
void* pool_get(int dev, size_t bytes, size_t* got) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int best = -1;
    for (int i = 0; i < (int) g_pool.size(); ++i)
        if (g_pool[i].dev == dev && g_pool[i].bytes >= bytes && g_pool[i].bytes <= 2 * bytes + (1u << 20) && (best < 0 || g_pool[i].bytes < g_pool[best].bytes)) best = i;
    if (best < 0) { *got = 0; return nullptr; }
    void* p = g_pool[best].p;
    *got = g_pool[best].bytes;
    g_pool_bytes -= g_pool[best].bytes;
    g_pool.erase(g_pool.begin() + best);
    return p;
}
void pool_put(int dev, void* p, size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (g_pool_bytes + bytes <= kPoolCap) { g_pool.push_back({p, bytes, dev}); g_pool_bytes += bytes; return; }
    }
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != dev) cudaSetDevice(dev);
    cudaFree(p);
    if (cur != dev) cudaSetDevice(cur);
}
size_t pool_release() {
    std::vector<PoolBlock> blocks;
    size_t n = 0;
    { std::lock_guard<std::mutex> lk(g_pool_mu); blocks.swap(g_pool); n = g_pool_bytes; g_pool_bytes = 0; }
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto& b : blocks) { cudaSetDevice(b.dev); cudaFree(b.p); }
    cudaSetDevice(cur);
    return n;
}

int twiddles2(int dev, int M, const float2** hi, const float2** lo) {
    struct Entry { int dev, M; float2 *hi, *lo; };
    static std::mutex mu;
    static std::vector<Entry> tab;
    std::lock_guard<std::mutex> lk(mu);
    for (auto& e : tab) if (e.dev == dev && e.M == M) { *hi = e.hi; *lo = e.lo; return 0; }
    const int nlo = 1024, nhi = (M + nlo - 1) / nlo;
    std::vector<float2> h(nhi + nlo);
    for (int a = 0; a < nhi; ++a) {
        const double ang = -2.0 * M_PI * ((double) a * nlo) / (double) M;
        h[a].x = (float) cos(ang); h[a].y = (float) sin(ang);
    }
    for (int b = 0; b < nlo; ++b) {
        const double ang = -2.0 * M_PI * (double) b / (double) M;
        h[nhi + b].x = (float) cos(ang); h[nhi + b].y = (float) sin(ang);
    }
    float2* d = nullptr;
    CK(cudaMalloc(&d, sizeof(float2) * h.size()));
    CK(cudaMemcpy(d, h.data(), sizeof(float2) * h.size(), cudaMemcpyHostToDevice));
    tab.push_back({dev, M, d, d + nhi});
    *hi = d; *lo = d + nhi;
    return 0;
}

}  // namespace irbh

namespace {

using irbh::fail;
using irbh::DevBuf;
using irbh::g_launches;

// FFT half-size M for a block size: N = smallest power of two >= 2B-1 (fp/convolution.cpp:45-48), M = N/2,
// never below 16 (a longer zero-padded transform gives the same linear convolution).
int half_size_for_block(int B) {
    int N = 1;
    while (N < 2 * B - 1) N *= 2;
    int M = N / 2;
    return M < 16 ? 16 : M;
}
constexpr int kMaxM = 2048;

// launch policy (irb_tuning.hpp): partitions per IR ring stage of the register-staged MAC (1 or 2), its FDL loads as 32-byte
// LDG.256 with L2 evict-first or 16-byte loads
int mac_u_pref() { return irbh::g_tuning.mac_u; }
bool mac_wide_pref() { return irbh::g_tuning.mac_wide != 0; }

template <int M>
int launch_fwd_t(const irb::FwdArgs& a, cudaStream_t st) {
    constexpr int R = irb::Tile<M>::ROWS;
    const int grid = (a.n_rows + R - 1) / R + (a.n_rr + R - 1) / R;
    if (grid <= 0) return 0;
    irb::k_fwd<M><<<grid, irb::kThreads, 0, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
// the non-persistent fused block step with the FDL streamed through TMA (k_mac_tma) or register-staged (k_mac<FUSE>)
bool mac_tma_pref() { return irbh::g_tuning.mac_tma != 0; }

// ---- persistent block step (irb_mac_p.cuh) ------------------------------------------------------------------------
constexpr int kPersistMinM = 256;
int persistent_ctas_per_sm() { const int c = irbh::g_tuning.persistent_ctas; return c >= 1 && c <= 2 ? c : 2; }
// Units of a launch over n_rows rows for `ctas` resident CTAs (fetch order: large units first).  Whole waves of full tiles,
// then the remainder rem < ROWS * ctas rows in t = ceil(rem / ctas) row-times: one wave of units of s rows for every set bit
// s of t (s = ROWS/2, ROWS/4 ...), so that a launch takes about ceil(n_rows / ctas) row-times instead of
// ceil(tiles / ctas) tile-times.  A unit of s rows starts at a multiple of s: it never straddles a tile.
void plan_units(int n_rows, int rows_per_tile, int ctas, bool narrowing, int out[4]) {
    out[0] = out[1] = out[2] = out[3] = 0;
    if (n_rows <= 0) return;
    const long long per_wave = (long long) rows_per_tile * ctas;
    const int waves = (int) (n_rows / per_wave);
    int rem = (int) (n_rows - waves * per_wave);
    out[0] = waves * ctas;
    if (rem == 0) return;
    const int t = (rem + ctas - 1) / ctas;                 // row-times the remainder needs at best
    if (!narrowing || rows_per_tile == 1 || t >= rows_per_tile) { out[0] += (rem + rows_per_tile - 1) / rows_per_tile; return; }
    int s = rows_per_tile / 2;
    for (int lvl = 1; lvl < 4 && s >= 1 && rem > 0; ++lvl, s /= 2) {
        if (!(t & s)) continue;
        const int cnt = std::min(ctas, (rem + s - 1) / s);
        out[lvl] = cnt;
        rem -= std::min(rem, cnt * s);
    }
}
// ---- per-device kernel set-up ------------------------------------------------------------------------------------------
// Cached per (kernel, device, key), not per thread: one thread drives every GPU of an irb_group, and a cache of its last device
// would redo the set-up on every switch.  Key 0: the attributes (kernel_setup); key n >= 1: the usable size of a requested
// cluster size n (launch_slots_t).
std::mutex g_setup_mu;
std::map<std::tuple<const void*, int, int>, int> g_setup;

// Once per (kernel, device): the dynamic shared memory `smem`, the largest shared-memory carveout if `max_carveout`, clusters
// above the portable size if `clusters`, and a check that `min_resident` CTAs fit on an SM (registers / shared memory): a
// kernel built for two CTAs per SM (ring depth, register budget) refuses to run silently at half of it.
int kernel_setup(const void* k, const char* name, int M, size_t smem, bool max_carveout, int min_resident, bool clusters = false) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_setup_mu);
    if (g_setup.count({k, dev, 0})) return 0;
    CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    if (max_carveout) CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (clusters) CK(cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    if (min_resident > 1) {
        int resident = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k, irb::kThreads + 32, smem));
        if (resident < min_resident)
            return fail(IRB_ERR_CUDA, "%s<%d>: only %d CTA per SM fits (registers / shared memory), %d expected", name, M, resident, min_resident);
    }
    g_setup[{k, dev, 0}] = 1;
    return 0;
}

// The persistent block steps: k_mac_p (INS == 0; irb_mac_p.cuh) over a.n_rows rows, or the IR-matrix step k_mac_mx
// (irb_mac_mx.cuh) over a.n_rows output rows in units of whole groups.  One launch, at most one CTA per unit.
template <int M, bool PER, int INS = 0, int OUTS = 0>
int launch_persistent(irb::MacArgs a, int num_sms, cudaStream_t st) {
    if (a.n_rows <= 0) return 0;
    if (!a.work) return fail(IRB_ERR_STATE, "persistent block step without a work counter");
    const int ctas = persistent_ctas_per_sm() * num_sms;
    void (*k)(irb::MacArgs);
    size_t smem;
    if constexpr (INS == 0) {
        plan_units(a.n_rows, irb::Tile<M>::ROWS, ctas, irbh::g_tuning.unit_narrowing != 0, a.unit_n);
        k = irb::k_mac_p<M, PER>;
        smem = sizeof(irb::PSmem<M, PER>);
    } else {
        using C = irb::MxCfg<M, INS, OUTS, PER>;
        a.unit_n[0] = (a.n_rows / OUTS + C::GROUPS - 1) / C::GROUPS; a.unit_n[1] = a.unit_n[2] = a.unit_n[3] = 0;
        k = irb::k_mac_mx<M, INS, OUTS, PER>;
        smem = sizeof(irb::MxSmem<M, INS, OUTS, PER>);
    }
    const int grid = std::min(a.unit_n[0] + a.unit_n[1] + a.unit_n[2] + a.unit_n[3], ctas);
    if (int rc = kernel_setup((const void*) k, INS == 0 ? "k_mac_p" : "k_mac_mx", M, smem, true, 2)) return rc;
    k<<<grid, irb::kThreads + 32, smem, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
template <int M, int INS, int OUTS>
int launch_mac_mx_pg(const irb::MacArgs& a, bool pergroup, int num_sms, cudaStream_t st) {
    return pergroup ? launch_persistent<M, true, INS, OUTS>(a, num_sms, st) : launch_persistent<M, false, INS, OUTS>(a, num_sms, st);
}
template <int M>
int launch_mac_mx_m(const irb::MacArgs& a, int ins, int outs, bool pergroup, int num_sms, cudaStream_t st) {
    if (ins == 1 && outs == 2) return launch_mac_mx_pg<M, 1, 2>(a, pergroup, num_sms, st);
    if (ins == 2 && outs == 2) return launch_mac_mx_pg<M, 2, 2>(a, pergroup, num_sms, st);
    return fail(IRB_ERR_ARG, "unsupported IR matrix %d x %d", ins, outs);
}
int launch_mac_mx(int M, int ins, int outs, bool pergroup, int num_sms, const irb::MacArgs& a, cudaStream_t st) {
    switch (M) {
        case 256: return launch_mac_mx_m<256>(a, ins, outs, pergroup, num_sms, st);
        case 512: return launch_mac_mx_m<512>(a, ins, outs, pergroup, num_sms, st);
        case 1024: return launch_mac_mx_m<1024>(a, ins, outs, pergroup, num_sms, st);
        default: return fail(IRB_ERR_ARG, "the matrix engine takes FFT half sizes 256 .. 1024, not %d", M);
    }
}
template <int M>
int launch_mac_tma(const irb::MacArgs& a, cudaStream_t st) {
    const int grid = (a.n_rows + irb::Tile<M>::ROWS - 1) / irb::Tile<M>::ROWS;
    if (grid <= 0) return 0;
    const size_t smem = sizeof(irb::TmaSmem<M>);
    if (int rc = kernel_setup((const void*) irb::k_mac_tma<M>, "k_mac_tma", M, smem, false, 0)) return rc;
    irb::k_mac_tma<M><<<grid, irb::kThreads + 32, smem, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
template <int M, int U, bool INV, bool FUSE = false, bool WIDE = false>
int launch_mac_u(const irb::MacArgs& a, cudaStream_t st) {
    const int grid = (a.n_rows + irb::Tile<M>::ROWS - 1) / irb::Tile<M>::ROWS;
    if (grid <= 0) return 0;
    const size_t smem = sizeof(irb::MacSmem<M, U>);
    if (int rc = kernel_setup((const void*) irb::k_mac<M, U, INV, FUSE, WIDE>, "k_mac", M, smem, false, 0)) return rc;
    irb::k_mac<M, U, INV, FUSE, WIDE><<<grid, irb::kThreads + 32, smem, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
// slot kernel: a.split_in slots per row inside a tile, clusters of `cl` CTAs splitting the partitions further
template <int M, bool INV>
int launch_slots_t(const irb::MacArgs& a, int cl, cudaStream_t st) {
    const int rpt = irb::Tile<M>::ROWS / a.split_in;
    const int tiles = (a.n_rows + rpt - 1) / rpt;
    if (tiles <= 0) return 0;
    const size_t smem = sizeof(irb::SlotSmem<M>);
    const void* k = (const void*) irb::k_mac_slots<M, INV>;
    if (int rc = kernel_setup(k, "k_mac_slots", M, smem, false, 0, true)) return rc;
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(irb::kThreads + 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    // the largest cluster this device can co-schedule, found once per (device, size): a partitioned or busy GPU may not
    // have 16 SMs free in one GPC; the kernel reads its cluster size at run time, so a smaller one just splits less
    int dev = 0;
    CK(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lk(g_setup_mu);
        int& usable = g_setup[{k, dev, cl}];
        if (usable == 0) {
            int c = cl;
            for (; c > 1; c /= 2) {
                cfg.gridDim = dim3((unsigned) c); at[0].val.clusterDim.x = (unsigned) c;
                int n = 0;
                if (cudaOccupancyMaxActiveClusters(&n, irb::k_mac_slots<M, INV>, &cfg) == cudaSuccess && n > 0) break;
                cudaGetLastError();
            }
            usable = c;
        }
        cl = usable;
    }
    cfg.gridDim = dim3((unsigned) (tiles * cl)); at[0].val.clusterDim.x = (unsigned) cl;
    CK(cudaLaunchKernelEx(&cfg, irb::k_mac_slots<M, INV>, a));
    g_launches++;
    return 0;
}
template <int M, bool INV>
int launch_mac_t(const irb::MacArgs& a, bool slots, int cl, int num_sms, cudaStream_t st) {
    if constexpr (INV && M >= kPersistMinM) {
        // the fused streaming block step as ONE persistent launch (shared-IR tiles or per-stream IRs)
        if (a.head && a.in && a.work && a.blocks_per_chan == 1 && a.head_back == 0 && a.split_in == 1 && cl == 1)
            return slots ? launch_persistent<M, true>(a, num_sms, st) : launch_persistent<M, false>(a, num_sms, st);
    }
    if (slots) return launch_slots_t<M, INV>(a, cl, st);
    if constexpr (INV) {
        if (a.head) {                                   // streaming block step
            if constexpr (M >= 256) { if (a.in && a.blocks_per_chan == 1 && mac_tma_pref()) return launch_mac_tma<M>(a, st); }
            if constexpr (M <= 512) {
                if (mac_wide_pref() && mac_u_pref() == 2) return a.in ? launch_mac_u<M, 2, true, true, true>(a, st) : launch_mac_u<M, 2, true, false, true>(a, st);
            }
            if (mac_wide_pref()) return a.in ? launch_mac_u<M, 1, true, true, true>(a, st) : launch_mac_u<M, 1, true, false, true>(a, st);
            if (a.in) return launch_mac_u<M, 1, true, true>(a, st);      // forward transform fused into the prologue
        }
    }
    if constexpr (!INV) { if (a.head && mac_wide_pref()) return launch_mac_u<M, 1, false, false, true>(a, st); }   // the bare MAC (measurement)
    if constexpr (M <= 512) { if (mac_u_pref() == 2) return launch_mac_u<M, 2, INV>(a, st); }
    return launch_mac_u<M, 1, INV>(a, st);
}
#define IRB_DISPATCH_M(M_, EXPR)                                         \
    switch (M_) {                                                        \
        case 16: { constexpr int MM = 16; return EXPR; }                 \
        case 32: { constexpr int MM = 32; return EXPR; }                 \
        case 64: { constexpr int MM = 64; return EXPR; }                 \
        case 128: { constexpr int MM = 128; return EXPR; }               \
        case 256: { constexpr int MM = 256; return EXPR; }               \
        case 512: { constexpr int MM = 512; return EXPR; }               \
        case 1024: { constexpr int MM = 1024; return EXPR; }             \
        case 2048: { constexpr int MM = 2048; return EXPR; }             \
        default: return fail(IRB_ERR_ARG, "unsupported FFT half size %d", M_); \
    }
int launch_fwd(int M, const irb::FwdArgs& a, cudaStream_t st) { IRB_DISPATCH_M(M, launch_fwd_t<MM>(a, st)); }
int launch_mac(int M, bool inv, bool slots, int cl, int num_sms, const irb::MacArgs& a, cudaStream_t st) {
    if (inv) { IRB_DISPATCH_M(M, (launch_mac_t<MM, true>(a, slots, cl, num_sms, st))); }
    IRB_DISPATCH_M(M, (launch_mac_t<MM, false>(a, slots, cl, num_sms, st)));
}
int tile_rows(int M) { return irb::kTile / M; }


}  // namespace

struct irb_engine {
    int device = 0, B = 0, M = 0, ring = 0, n_chans = 0, n_irs = 0;
    int active = 0;                    // channels [0, active) take part in a block step (irb_engine_set_active_channels); I/O arrays are dense over them
    // IR-matrix engine (irb_engine_create_matrix): groups of `ins` input channels producing `outs` output channels each.  The
    // channels above (n_chans, active, FDL rows, heads) are the INPUTS; ov and the output staging hold n_chans / ins * outs
    // rows; h_ir_of_chan / ir_of_chan hold the matrix table [group][ins * outs]; per_row_ir means "some unit mixes matrices".
    // A plain engine is the 1 x 1 case.
    int ins = 1, outs = 1;
    bool matrix() const { return ins != 1 || outs != 1; }
    int out_chans() const { return active / ins * outs; }
    size_t in_blk() const { return (size_t) B * active; }
    size_t out_blk() const { return (size_t) B * out_chans(); }
    // FDL layout [chan / fdl_group][slot][chan % fdl_group][M], fdl_group = channels per kernel tile (irb_kernels.cuh, MacArgs)
    int fdl_group = 1;
    long long fdl_group_stride() const { return (long long) ring * fdl_group * M; }
    size_t fdl_bytes() const { return sizeof(float2) * (size_t) ((n_chans + fdl_group - 1) / fdl_group) * (size_t) fdl_group_stride(); }
    cudaStream_t own_stream = nullptr, stream = nullptr;
    const float2* W = nullptr;
    DevBuf fdl, H, ov, head, ir_of_chan, nparts, io_in[2], io_out[2], taps;
    // IR loads (irb_engine_set_irs / _stage_irs): the item table of k_ir_load, grown on demand; the pooled staging of a load from
    // host memory larger than `taps`, held until the load is waited for; upload / transform events of its two staging slots
    DevBuf ld_tab;
    size_t ld_tab_cap = 0;
    std::unique_ptr<irbh::ScratchBuf> ld_stage;
    cudaEvent_t ld_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    DevBuf work;                       // k_mac_p: {next unit, finished CTAs}, cleared by the kernel itself
    unsigned long long* stamps = nullptr;   // measurement only (irbx_engine_set_stamps): phase time stamps of the latency-path kernel
    int h_reps = 1;                    // identical copies of the IR spectra H (MacArgs::h_reps): [rep][ir][partition][M]
    long long h_rep_stride() const { return (long long) n_irs * ring * M; }
    // clear the spectra of one IR in every copy
    int ir_clear_all(int ir, cudaStream_t st) {
        for (int r = 0; r < h_reps; ++r) CK(cudaMemsetAsync(H.as<float2>() + r * h_rep_stride() + (size_t) ir * ring * M, 0, sizeof(float2) * (size_t) M * ring, st));
        return 0;
    }
    std::vector<int> h_ir_of_chan, h_nparts;
    bool binding_dirty = true;
    bool per_row_ir = false;           // some kernel tile mixes IRs: every slot stages its own IR partitions (k_mac_slots)
    // launch plan of the MAC (recomputed when bindings or IR lengths change): with few rows the partitions of a row
    // are split over split_in slots of a tile and cluster_dim CTAs of a cluster (k_mac_slots)
    bool plan_dirty = true;
    int split_in = 1, cluster_dim = 1;
    int force_split_in = 0, force_cluster = 0;      // irb_engine_set_mac_split
    bool fuse_fwd = true;                           // irb_engine_set_fused_step
    int num_sms = 148;
    // round-robin IR refresh (Source/PluginProcessor.cpp:455-461): staged taps per IR, positions on the device
    std::vector<std::unique_ptr<DevBuf>> rr_buf;
    std::vector<int> h_rr_list;
    DevBuf rr_ptrs, rr_pos, rr_list;
    std::unique_ptr<DevBuf> cb_in, cb_out;          // irb_engine_process_callback staging, grown on demand
    int cb_blocks = 0;
    // The latency path (one small block per call): copy-in, the step's kernels and copy-out are captured ONCE into a CUDA
    // graph over pinned staging owned by the engine and replayed with a single launch per block.  The signature records
    // everything the captured launches baked in; a change re-captures.
    struct GraphSig { int n_rr, split_in, cluster, slots, fuse, active, variant; cudaStream_t stream; int in_fmt, out_fmt; bool operator==(const GraphSig& o) const {
        return n_rr == o.n_rr && split_in == o.split_in && cluster == o.cluster && slots == o.slots && fuse == o.fuse && active == o.active &&
               variant == o.variant && stream == o.stream && in_fmt == o.in_fmt && out_fmt == o.out_fmt; } };
    cudaGraphExec_t g_exec = nullptr;
    GraphSig g_sig{-1, 0, 0, 0, 0, 0, 0, nullptr, 0, 0};
    void *g_hin = nullptr, *g_hout = nullptr;
    int g_kernels = 0;
    bool g_warm = false;                             // a plain step with this signature has run (kernel attributes are set)
    bool use_graph = true;
    size_t bytes = 0;
    long long launches = 0;
    // host path: copy streams + events so block b+1 uploads and block b-1 downloads while block b computes
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    // optional per-step device timing: events before k_fwd, before k_mac, after k_mac
    bool timing = false;
    std::vector<cudaEvent_t> tev;
    std::vector<char> tev_mid;                           // step i recorded its middle event (a kernel ran before the MAC launch)
    int t_rec = 0;
    std::vector<cudaEvent_t> ev_grp;                 // single large block: per channel group "uploaded" / "computed"
    unsigned long long pipe_seq = 0;                 // blocks that went through the multi-block pipeline (staging slot = seq & 1)
    bool pipe_pending = false;                       // submitted work not yet waited for
    ~irb_engine() {
        for (auto ev : tev) cudaEventDestroy(ev);
        for (auto ev : ev_grp) if (ev) cudaEventDestroy(ev);
        for (auto ev : ld_ev) if (ev) cudaEventDestroy(ev);
        for (int i = 0; i < 2; ++i) {
            if (ev_in[i]) cudaEventDestroy(ev_in[i]);
            if (ev_done[i]) cudaEventDestroy(ev_done[i]);
            if (ev_out[i]) cudaEventDestroy(ev_out[i]);
        }
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
        if (g_exec) cudaGraphExecDestroy(g_exec);
        if (g_hin) cudaFreeHost(g_hin);
        if (g_hout) cudaFreeHost(g_hout);
    }
};

namespace {

int floor_pow2(long long x) { int r = 1; while (2LL * r <= x) r *= 2; return r; }

int engine_check_binding(irb_engine* e) {
    if (e->matrix()) {
        // one launch of k_mac_mx per step, no partition split; PERGROUP when some unit's groups are bound to different matrices
        if (e->binding_dirty) {
            const int terms = e->ins * e->outs, n_groups = e->n_chans / e->ins;
            const int per_unit = tile_rows(e->M) / e->outs;
            e->per_row_ir = false;
            for (int g = 0; g < n_groups && !e->per_row_ir; ++g)
                if (g % per_unit && !std::equal(e->h_ir_of_chan.begin() + (size_t) g * terms, e->h_ir_of_chan.begin() + (size_t) (g + 1) * terms,
                                                e->h_ir_of_chan.begin() + (size_t) (g - g % per_unit) * terms)) e->per_row_ir = true;
            CK(cudaMemcpyAsync(e->ir_of_chan.p, e->h_ir_of_chan.data(), sizeof(int) * e->h_ir_of_chan.size(), cudaMemcpyHostToDevice, e->stream));
            CK(cudaStreamSynchronize(e->stream));
            e->binding_dirty = false;
        }
        e->split_in = 1; e->cluster_dim = 1; e->plan_dirty = false;
        return 0;
    }
    if (e->binding_dirty) {
        const int rows = tile_rows(e->M);
        e->per_row_ir = false;
        for (int c0 = 0; c0 < e->n_chans && !e->per_row_ir; c0 += rows)
            for (int c = c0 + 1; c < c0 + rows && c < e->n_chans; ++c)
                if (e->h_ir_of_chan[c] != e->h_ir_of_chan[c0]) { e->per_row_ir = true; break; }
        CK(cudaMemcpyAsync(e->ir_of_chan.p, e->h_ir_of_chan.data(), sizeof(int) * e->n_chans, cudaMemcpyHostToDevice, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        e->binding_dirty = false;
        e->plan_dirty = true;
    }
    if (e->plan_dirty) {
        // Few rows: fill the GPU by splitting each row's partitions.  Target two CTAs per SM; at least 4 partitions
        // per slot; the reduced tile (1024/split_in float4) must divide among the CTAs of a cluster.
        const int rows = tile_rows(e->M);
        const int tiles = (e->active + rows - 1) / rows;
        int split_in = 1, cl = 1;
        if (tiles * 2 <= e->num_sms) {
            int max_np = 1;
            for (int c = 0; c < e->active; ++c) max_np = std::max(max_np, e->h_nparts[e->h_ir_of_chan[c]]);
            long long want = floor_pow2(std::max<long long>(1, 2LL * e->num_sms * rows / e->active));
            want = std::min<long long>(want, floor_pow2(std::max(1, max_np / 4)));
            split_in = (int) std::min<long long>(want, rows);
            cl = (int) std::min<long long>(want / split_in, 16);
        }
        if (e->force_split_in > 0) { split_in = e->force_split_in; cl = e->force_cluster; }
        split_in = std::max(1, std::min(floor_pow2(split_in), rows));
        cl = std::max(1, std::min(floor_pow2(cl), std::min(16, 1024 / split_in)));
        e->split_in = split_in; e->cluster_dim = cl;
        e->plan_dirty = false;
    }
    return 0;
}

// the ring-protocol knobs every MAC launch carries (irb_tuning.hpp)
void mac_policy(irb::MacArgs& m) {
    m.producer_sleep_ns = irbh::g_tuning.producer_sleep_ns;
    m.release_fence = irbh::g_tuning.release_fence;
    m.release_dep = irbh::g_tuning.release_dep;
}

// Every launch helper takes a channel range [c0, c0 + cn): all per-channel arrays are offset, so a kernel sees rows
// 0 .. cn-1.  c0 is a multiple of the tile's row count (tiles never straddle a range).
void fill_mac_args(irb_engine* e, irb::MacArgs& m, int c0, int cn) {
    m.fdl = e->fdl.as<float2>() + (size_t) (c0 / e->fdl_group) * e->fdl_group_stride(); m.fdl_chan_stride = e->fdl_group_stride();
    m.fdl_group = e->fdl_group; m.fdl_slot_stride = (long long) e->fdl_group * e->M;
    m.head = e->head.as<int>() + c0; m.ring = e->ring; m.blocks_per_chan = 1; m.n_rows = cn;
    m.H = e->H.as<float2>(); m.ir_stride = (long long) e->ring * e->M;
    m.h_reps = e->h_reps; m.h_rep_stride = e->h_rep_stride(); m.stagger_ns = irbh::g_tuning.stagger_ns; m.ring_stages = irbh::g_tuning.ring_stages;
    m.ir_of_chan = e->ir_of_chan.as<int>() + c0; m.nparts = e->nparts.as<int>(); m.W = e->W;
    m.B = e->B; m.split_in = e->split_in;
    mac_policy(m);
    m.stamps = e->stamps;
    m.work = irbh::g_tuning.mac_persistent ? e->work.as<int>() : nullptr;
}
bool use_slots(const irb_engine* e) { return e->per_row_ir || e->split_in > 1 || e->cluster_dim > 1; }
// Is the block step ONE launch (forward transform in the MAC kernel's prologue)?  Shared-IR tiles: always (unless switched off);
// per-stream IRs: through the persistent kernel; few rows (partitions split over slots / a cluster): in the cluster kernel.
bool step_is_fused(const irb_engine* e) {
    if (e->matrix()) return true;                   // k_mac_mx always transforms the new blocks itself
    if (!e->fuse_fwd) return false;
    if (e->split_in > 1 || e->cluster_dim > 1) return irbh::g_tuning.fuse_split != 0;      // the cluster kernel's rank 0 transforms the new blocks itself
    if (e->per_row_ir) return irbh::g_tuning.mac_persistent && e->M >= kPersistMinM;
    return true;
}
// everything a captured graph or a cached plan bakes in besides the engine's own state
int tuning_variant() {
    const irbh::Tuning& t = irbh::g_tuning;
    return t.mac_persistent | t.mac_tma << 1 | t.mac_wide << 2 | (t.mac_u & 3) << 3 | t.release_fence << 5 | t.release_dep << 9 | t.fuse_split << 10 | (t.persistent_ctas & 3) << 6 | t.unit_narrowing << 8;
}

constexpr int kTimingCap = 16384;

// the sample format of a block array (irb_sample_format): element size, and the address of element i
bool fmt_valid(int fmt) { return fmt == IRB_SAMPLE_F32 || fmt == IRB_SAMPLE_S16 || fmt == IRB_SAMPLE_S24; }
size_t fmt_size(int fmt) { return (size_t) irb::fmt_bytes(fmt); }
template <class T> T* fmt_at(T* p, int fmt, size_t i) {
    using Byte = typename std::conditional<std::is_const<T>::value, const unsigned char, unsigned char>::type;
    return p ? (T*) ((Byte*) p + i * fmt_size(fmt)) : nullptr;
}

// forward FFT of one block of the channels of the range into the FDL (advances their heads) and/or the round-robin IR
// refresh rows; in_dev / out_dev below are the block's arrays for ALL channels, in the formats in_fmt / out_fmt
int engine_launch_fwd(irb_engine* e, const void* in_dev, int in_fmt, bool audio, bool refresh, int c0, int cn) {
    irb::FwdArgs f{};
    f.src = fmt_at(in_dev, in_fmt, (size_t) c0 * e->B); f.src_fmt = in_fmt; f.src2 = nullptr; f.src_chan_stride = e->B; f.L = e->B; f.B = e->B;
    f.blocks_per_chan = 1; f.n_rows = audio ? cn : 0;
    f.dst = e->fdl.as<float2>() + (size_t) (c0 / e->fdl_group) * e->fdl_group_stride(); f.dst_chan_stride = e->fdl_group_stride();
    f.dst_group = e->fdl_group; f.dst_slot_stride = (long long) e->fdl_group * e->M;
    f.head = e->head.as<int>() + c0; f.ring = e->ring; f.W = e->W;
    // one IR partition of every staged IR is re-transformed per block, in the same launch
    f.n_rr = refresh ? (int) e->h_rr_list.size() : 0; f.rr_list = e->rr_list.as<int>(); f.rr_taps = e->rr_ptrs.as<const float*>();
    f.rr_pos = e->rr_pos.as<int>(); f.nparts = e->nparts.as<int>(); f.H = e->H.as<float2>(); f.ir_stride = (long long) e->ring * e->M;
    f.h_reps = e->h_reps; f.h_rep_stride = e->h_rep_stride();
    if (f.n_rows == 0 && f.n_rr == 0) return 0;
    int rc = launch_fwd(e->M, f, e->stream);
    if (rc) return rc;
    e->launches += 1;
    return 0;
}
// the IR-matrix block step over every group: inputs in_dev [n_chans][B], outputs out_dev [n_chans / ins * outs][B]
int engine_launch_mx(irb_engine* e, void* out_dev, int out_fmt, const void* in_dev, int in_fmt) {
    irb::MacArgs m{};
    fill_mac_args(e, m, 0, e->n_chans);
    m.n_rows = e->out_chans(); m.work = e->work.as<int>();
    m.Y = nullptr; m.out = out_dev; m.out_fmt = out_fmt; m.out_chan_stride = e->B; m.Lout = e->B;
    m.ov = e->ov.as<float>(); m.tail = nullptr; m.head_back = 0;
    m.in = in_dev; m.in_fmt = in_fmt; m.in_chan_stride = e->B; m.head_rw = e->head.as<int>();
    int rc = launch_mac_mx(e->M, e->ins, e->outs, e->per_row_ir, e->num_sms, m, e->stream);
    if (rc) return rc;
    e->launches += 1;
    return 0;
}
// in_dev != nullptr: the forward transform of that block runs inside the MAC kernel (shared-IR kernel only)
int engine_launch_mac(irb_engine* e, void* out_dev, int out_fmt, int head_back, const void* in_dev, int in_fmt, int c0, int cn) {
    if (e->matrix()) return engine_launch_mx(e, out_dev, out_fmt, in_dev, in_fmt);
    irb::MacArgs m{};
    fill_mac_args(e, m, c0, cn);
    m.Y = nullptr; m.out = fmt_at(out_dev, out_fmt, (size_t) c0 * e->B); m.out_fmt = out_fmt; m.out_chan_stride = e->B; m.Lout = e->B;
    m.ov = e->ov.as<float>() + (size_t) c0 * e->B; m.tail = nullptr; m.head_back = head_back;
    m.in = fmt_at(in_dev, in_fmt, (size_t) c0 * e->B); m.in_fmt = in_fmt; m.in_chan_stride = e->B; m.head_rw = e->head.as<int>() + c0;
    int rc = launch_mac(e->M, true, use_slots(e), e->cluster_dim, e->num_sms, m, e->stream);
    if (rc) return rc;
    e->launches += 1;
    return 0;
}

// one block step for the channels [c0, c0+cn); refresh: also run the staged IRs' refresh rows (once per block)
int engine_step_range(irb_engine* e, const void* in_dev, int in_fmt, void* out_dev, int out_fmt, int c0, int cn, bool refresh) {
    // ONE launch per block step, the forward transform is the MAC kernel's prologue (staged IRs still get their refresh
    // rows through a k_fwd launch of their own).  The few-row cluster kernel transforms the new blocks on its rank 0.
    const bool fused = step_is_fused(e);
    int rc = engine_launch_fwd(e, in_dev, in_fmt, !fused, refresh, c0, cn);
    if (rc) return rc;
    return engine_launch_mac(e, out_dev, out_fmt, 0, fused ? in_dev : nullptr, in_fmt, c0, cn);
}

int engine_step_device(irb_engine* e, const void* in_dev, int in_fmt, void* out_dev, int out_fmt) {
    const bool rec = e->timing && e->t_rec < kTimingCap;
    if (rec) CK(cudaEventRecord(e->tev[3 * e->t_rec], e->stream));
    const bool fused = step_is_fused(e);
    const long long launched = g_launches.load();
    int rc = engine_launch_fwd(e, in_dev, in_fmt, !fused, true, 0, e->active);
    if (rc) return rc;
    // the middle event only where a kernel ran before the MAC launch: on a one-launch step it would add its own 2-3 us to the step
    const bool mid = rec && g_launches.load() != launched;
    if (rec) e->tev_mid[e->t_rec] = mid;
    if (mid) CK(cudaEventRecord(e->tev[3 * e->t_rec + 1], e->stream));
    if ((rc = engine_launch_mac(e, out_dev, out_fmt, 0, fused ? in_dev : nullptr, in_fmt, 0, e->active))) return rc;
    if (rec) { CK(cudaEventRecord(e->tev[3 * e->t_rec + 2], e->stream)); e->t_rec++; }
    return 0;
}

}  // namespace

extern "C" {

const char* irb_last_error(void) { return irbh::g_err; }
int irb_version(void) { return 100; }
int irb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return fail(IRB_ERR_CUDA, "no CUDA device"); }
    return n;
}
int irb_set_device(int device) {
    CK(cudaSetDevice(device));
    irbh::g_device = device;
    return 0;
}
int irb_max_block_size(void) { return kMaxM; }
void* irb_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 16) != cudaSuccess) { cudaGetLastError(); fail(IRB_ERR_CUDA, "cudaMallocHost(%zu) failed", bytes); return nullptr; }
    return p;
}
void* irb_host_alloc_write_combined(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocWriteCombined) != cudaSuccess) { cudaGetLastError(); fail(IRB_ERR_CUDA, "cudaHostAlloc(%zu, write-combined) failed", bytes); return nullptr; }
    return p;
}
void irb_host_free(void* p) { if (p) cudaFreeHost(p); }
long long irb_launch_count(void) { return g_launches.load(); }
size_t irb_release_workspace(void) { return irbh::pool_release(); }
double irb_last_compute_ms(void) { return irbh::g_last_compute_ms; }

}  // extern "C"
namespace {
// n_channels INPUT channels; a matrix engine (ins x outs != 1 x 1) has n_channels / ins groups and n_channels / ins * outs outputs
int engine_create(irb_engine** out, int device, int block_size, int max_partitions, int n_channels, int n_irs, int ins, int outs) {
    CK(cudaSetDevice(device));
    irb_engine* e = new (std::nothrow) irb_engine;
    if (!e) return fail(IRB_ERR_ARG, "out of host memory");
    e->device = device; e->B = block_size; e->M = half_size_for_block(block_size);
    e->ring = max_partitions; e->n_chans = n_channels; e->active = n_channels; e->n_irs = n_irs;
    e->ins = ins; e->outs = outs;
    const int n_out = n_channels / ins * outs, n_table = n_channels / ins * ins * outs;     // output rows; ir_of_chan entries
    int rc = irbh::twiddles(device, e->M, &e->W);
    if (rc) { delete e; return rc; }
    const size_t spec = sizeof(float2) * (size_t) e->M;
    // A/B: [chan][slot][M] instead of the tile-interleaved layout.  A matrix engine interleaves the input rows of one unit of its kernel.
    e->fdl_group = irbh::g_tuning.fdl_plain ? 1 : (e->matrix() ? tile_rows(e->M) / outs * ins : tile_rows(e->M));
    // shared IR spectra in several identical copies (MacArgs::h_reps): as many as fit 24 MB, at most 32; one when the IRs are many
    {
        const size_t one = spec * e->ring * n_irs;
        const int pref = irbh::g_tuning.ir_replicas;
        e->h_reps = pref > 0 ? std::min(pref, 64) : (int) std::max<size_t>(1, std::min<size_t>(32, (24u << 20) / one));
    }
    const size_t b_fdl = e->fdl_bytes(), b_H = spec * e->ring * n_irs * e->h_reps, b_io = sizeof(float) * (size_t) e->B * n_channels;
    const size_t b_oo = sizeof(float) * (size_t) e->B * n_out;
    if ((rc = e->fdl.alloc(b_fdl, true)) || (rc = e->H.alloc(b_H, true)) || (rc = e->ov.alloc(b_oo, true)) ||
        (rc = e->head.alloc(sizeof(int) * n_channels, false)) || (rc = e->ir_of_chan.alloc(sizeof(int) * n_table, true)) ||
        (rc = e->nparts.alloc(sizeof(int) * n_irs, true)) || (rc = e->io_in[0].alloc(b_io, true)) || (rc = e->io_out[0].alloc(b_oo, true)) ||
        (rc = e->io_in[1].alloc(b_io, true)) || (rc = e->io_out[1].alloc(b_oo, true)) ||
        (rc = e->taps.alloc(sizeof(float) * 2 * (size_t) e->B * e->ring, true)) || (rc = e->rr_ptrs.alloc(sizeof(float*) * n_irs, true)) ||
        (rc = e->rr_pos.alloc(sizeof(int) * n_irs, true)) || (rc = e->rr_list.alloc(sizeof(int) * n_irs, true)) || (rc = e->work.alloc(sizeof(int) * 4, true))) {
        delete e;
        return rc;
    }
    e->rr_buf.resize(n_irs);
    if (cudaDeviceGetAttribute(&e->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || e->num_sms < 1) { cudaGetLastError(); e->num_sms = 148; }
    e->bytes = b_fdl + b_H + 2 * b_io + 3 * b_oo + sizeof(int) * ((size_t) n_channels + n_table + 3 * (size_t) n_irs) + sizeof(float*) * n_irs + sizeof(float) * 2 * (size_t) e->B * e->ring;
    e->h_ir_of_chan.assign(n_table, 0);
    for (int i = 0; i < n_table; ++i) e->h_ir_of_chan[i] = i % (ins * outs);        // matrix: every group starts on IRs 0 .. ins*outs-1
    e->h_nparts.assign(n_irs, 0);
    bool ok = cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
        ok = cudaEventCreateWithFlags(&e->ev_in[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&e->ev_done[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&e->ev_out[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { delete e; return fail(IRB_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError())); }
    e->stream = e->own_stream;
    *out = e;
    return irb_engine_reset(e);
}
}  // namespace
extern "C" {

int irb_engine_create(irb_engine** out, int device, int block_size, int max_partitions, int n_channels, int n_irs) {
    if (!out) return fail(IRB_ERR_ARG, "out is null");
    *out = nullptr;
    if (block_size < 1 || half_size_for_block(block_size) > kMaxM) return fail(IRB_ERR_ARG, "block_size %d outside [1, %d]", block_size, kMaxM);
    if (max_partitions < 1 || n_channels < 1 || n_irs < 1) return fail(IRB_ERR_ARG, "max_partitions, n_channels and n_irs must be >= 1");
    return engine_create(out, device, block_size, max_partitions, n_channels, n_irs, 1, 1);
}

int irb_engine_create_matrix(irb_engine** out, int device, int block_size, int max_partitions, int n_groups, int ins, int outs, int n_irs) {
    if (!out) return fail(IRB_ERR_ARG, "out is null");
    *out = nullptr;
    if (!((ins == 1 && outs == 2) || (ins == 2 && outs == 2))) return fail(IRB_ERR_ARG, "IR matrix %d x %d: only 1 x 2 (mono -> stereo) and 2 x 2 (true stereo) exist", ins, outs);
    if (block_size < 129 || block_size > 1024) return fail(IRB_ERR_ARG, "block_size %d outside [129, 1024] (FFT half sizes 256 .. 1024)", block_size);
    if (max_partitions < 1 || n_groups < 1) return fail(IRB_ERR_ARG, "max_partitions and n_groups must be >= 1");
    if (n_irs < ins * outs) return fail(IRB_ERR_ARG, "n_irs %d is fewer than the %d IRs of one matrix", n_irs, ins * outs);
    if ((long long) n_groups * (ins > outs ? ins : outs) > 0x7fffffffLL / 2048) return fail(IRB_ERR_ARG, "n_groups %d too large", n_groups);
    return engine_create(out, device, block_size, max_partitions, n_groups * ins, n_irs, ins, outs);
}

int irb_engine_bind_matrix(irb_engine* e, int group_begin, int group_end, const int* ir_ids) {
    if (!e || !ir_ids) return fail(IRB_ERR_ARG, "engine or ir_ids null");
    if (!e->matrix()) return fail(IRB_ERR_STATE, "a plain engine binds channels: use irb_engine_bind");
    const int n_groups = e->n_chans / e->ins, terms = e->ins * e->outs;
    if (group_begin < 0 || group_end > n_groups || group_begin > group_end) return fail(IRB_ERR_ARG, "group range [%d, %d) outside [0, %d)", group_begin, group_end, n_groups);
    for (int t = 0; t < terms; ++t)
        if (ir_ids[t] < 0 || ir_ids[t] >= e->n_irs) return fail(IRB_ERR_ARG, "ir_ids[%d] = %d outside [0, %d)", t, ir_ids[t], e->n_irs);
    for (int g = group_begin; g < group_end; ++g)
        for (int t = 0; t < terms; ++t) e->h_ir_of_chan[(size_t) g * terms + t] = ir_ids[t];
    e->binding_dirty = true;
    return 0;
}

int irb_engine_destroy(irb_engine* e) {
    if (!e) return 0;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
    return 0;
}

int irb_engine_set_stream(irb_engine* e, void* cuda_stream) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream == IRB_OWN_STREAM ? e->own_stream : (cudaStream_t) cuda_stream;
    return 0;
}

int irb_engine_reset(irb_engine* e) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    CK(cudaMemsetAsync(e->fdl.p, 0, e->fdl_bytes(), e->stream));
    CK(cudaMemsetAsync(e->ov.p, 0, sizeof(float) * (size_t) e->B * (e->n_chans / e->ins * e->outs), e->stream));
    std::vector<int> h(e->n_chans, e->ring - 1);     // first block lands in slot 0
    CK(cudaMemcpyAsync(e->head.p, h.data(), sizeof(int) * e->n_chans, cudaMemcpyHostToDevice, e->stream));
    // staged IRs start over like irFftBufferArray.clearAndResize in prepareToPlay (PluginProcessor.cpp:226): spectra
    // cleared, write position 0; their partitions come back one per block
    for (int ir : e->h_rr_list) { int rc = e->ir_clear_all(ir, e->stream); if (rc) return rc; }
    CK(cudaMemsetAsync(e->rr_pos.p, 0, sizeof(int) * e->n_irs, e->stream));
    CK(cudaMemsetAsync(e->work.p, 0, sizeof(int) * 4, e->stream));          // the persistent kernel's unit counter (it clears itself; belt and braces)
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// One-row calls of irb_engine_set_irs / _stage_irs (their checks, their launch; same results and errors as ever).
int irb_engine_set_ir(irb_engine* e, int ir_id, const float* left, const float* right, int n_taps) {
    return irb_engine_set_irs(e, 1, &ir_id, left, right, n_taps, &n_taps);
}

// "IRtoConvolve = this buffer" (PluginProcessor.cpp:411-414): nothing is transformed here; every following block step
// re-transforms ONE partition of the staged taps, round-robin (:455-461), so a new IR replaces the old one partition
// by partition over nparts blocks.  The first call for an IR fixes its partition count (n_partitions, or
// ceil(n_taps / block_size) when 0) and starts from cleared spectra, as prepareToPlay does (:225-226).
int irb_engine_stage_ir(irb_engine* e, int ir_id, const float* left, const float* right, int n_taps, int n_partitions) {
    return irb_engine_stage_irs(e, 1, &ir_id, left, right, n_taps, &n_taps, n_partitions);
}

int irb_engine_bind(irb_engine* e, int chan_begin, int chan_end, int ir_id) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    if (e->matrix()) return fail(IRB_ERR_STATE, "an IR-matrix engine binds whole groups: use irb_engine_bind_matrix");
    if (chan_begin < 0 || chan_end > e->n_chans || chan_begin > chan_end) return fail(IRB_ERR_ARG, "channel range [%d, %d) outside [0, %d)", chan_begin, chan_end, e->n_chans);
    if (ir_id < 0 || ir_id >= e->n_irs) return fail(IRB_ERR_ARG, "ir_id %d outside [0, %d)", ir_id, e->n_irs);
    for (int c = chan_begin; c < chan_end; ++c) e->h_ir_of_chan[c] = ir_id;
    e->binding_dirty = true;
    return 0;
}
int irb_engine_tile_channels(const irb_engine* e) { return e ? tile_rows(e->M) : fail(IRB_ERR_ARG, "engine is null"); }
int irb_engine_set_mac_split(irb_engine* e, int split_in, int cluster) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    if (e->matrix()) return fail(IRB_ERR_STATE, "an IR-matrix engine has no partition split: its block step is one k_mac_mx launch");
    if (split_in < 0 || cluster < 0 || (split_in == 0) != (cluster == 0)) return fail(IRB_ERR_ARG, "split_in and cluster must both be 0 (automatic) or both >= 1");
    e->force_split_in = split_in; e->force_cluster = cluster;
    e->plan_dirty = true;
    return 0;
}
int irb_engine_set_fused_step(irb_engine* e, int enable) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    if (e->matrix() && !enable) return fail(IRB_ERR_STATE, "an IR-matrix engine has no two-launch form: its block step always transforms the new blocks itself");
    e->fuse_fwd = enable != 0;
    return 0;
}
int irb_engine_mac_plan(irb_engine* e, int* slots_kernel, int* split_in, int* cluster) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    int rc = engine_check_binding(e);
    if (rc) return rc;
    if (slots_kernel) *slots_kernel = use_slots(e) ? 1 : 0;
    if (split_in) *split_in = e->split_in;
    if (cluster) *cluster = e->cluster_dim;
    return 0;
}

int irb_engine_process_device(irb_engine* e, const float* in_dev, float* out_dev, int n_blocks) {
    return irb_engine_process_device_pcm(e, in_dev, IRB_SAMPLE_F32, out_dev, IRB_SAMPLE_F32, n_blocks);
}
int irb_engine_process_device_pcm(irb_engine* e, const void* in_dev, int in_format, void* out_dev, int out_format, int n_blocks) {
    if (!fmt_valid(in_format) || !fmt_valid(out_format)) return fail(IRB_ERR_ARG, "sample format %d / %d is not an irb_sample_format", in_format, out_format);
    if (!e || !in_dev || !out_dev) return fail(IRB_ERR_ARG, "null argument");
    if (n_blocks < 0) return fail(IRB_ERR_ARG, "n_blocks < 0");
    CK(cudaSetDevice(e->device));
    int rc = engine_check_binding(e);
    if (rc) return rc;
    const size_t iblk = e->in_blk(), oblk = e->out_blk();
    for (int b = 0; b < n_blocks; ++b)
        if ((rc = engine_step_device(e, fmt_at(in_dev, in_format, b * iblk), in_format, fmt_at(out_dev, out_format, b * oblk), out_format))) return rc;
    return 0;
}

namespace {
constexpr size_t kGraphMaxBytes = 256 << 10;         // blocks up to this size take the captured-graph path
constexpr int kMaxGroups = 16;                       // channel groups a large single block is pipelined over

// one block, host to host, as a single graph launch; *done = false when the caller should take the plain path instead.
// Matrix engines take this path too: input and output staging are sized by their own channel counts.
// The pinned staging holds kGraphMaxBytes whatever the formats; the eligibility test is made at float size, so a change of
// format never changes which path a block takes, only the captured byte counts (the signature holds both formats).
int engine_process_one_graphed(irb_engine* e, const void* in_host, int in_fmt, void* out_host, int out_fmt, bool* done) {
    *done = false;
    if (irbh::g_tuning.no_graph || !e->use_graph || e->timing || sizeof(float) * std::max(e->in_blk(), e->out_blk()) > kGraphMaxBytes) return 0;
    const size_t bytes = fmt_size(in_fmt) * e->in_blk(), obytes = fmt_size(out_fmt) * e->out_blk();      // (differ on a matrix engine)
    const irb_engine::GraphSig sig{(int) e->h_rr_list.size(), e->split_in, e->cluster_dim, use_slots(e) ? 1 : 0, e->fuse_fwd ? 1 : 0, e->active, tuning_variant(), e->stream,
                                   in_fmt, out_fmt};
    if (!(sig == e->g_sig)) {
        if (e->g_exec) { cudaGraphExecDestroy(e->g_exec); e->g_exec = nullptr; }
        e->g_sig = sig;
        e->g_warm = false;
    }
    if (!e->g_warm) { e->g_warm = true; return 0; }          // first block with this signature runs plainly
    if (!e->g_exec) {
        if (!e->g_hin) { CK(cudaMallocHost(&e->g_hin, kGraphMaxBytes)); CK(cudaMallocHost(&e->g_hout, kGraphMaxBytes)); }
        const long long l0 = e->launches;
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeRelaxed));
        int rc = cudaMemcpyAsync(e->io_in[0].p, e->g_hin, bytes, cudaMemcpyHostToDevice, e->stream) == cudaSuccess ? 0 : IRB_ERR_CUDA;
        if (!rc) rc = engine_step_device(e, e->io_in[0].p, in_fmt, e->io_out[0].p, out_fmt);
        if (!rc && cudaMemcpyAsync(e->g_hout, e->io_out[0].p, obytes, cudaMemcpyDeviceToHost, e->stream) != cudaSuccess) rc = IRB_ERR_CUDA;
        const cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
        e->g_kernels = (int) (e->launches - l0);
        e->launches = l0;                                    // nothing ran yet
        g_launches -= e->g_kernels;
        if (rc || ce != cudaSuccess || !graph) {             // capture refused: fall back to plain launches for good
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            e->use_graph = false;
            return 0;
        }
        const cudaError_t ie = cudaGraphInstantiate(&e->g_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); e->g_exec = nullptr; e->use_graph = false; return 0; }
    }
    memcpy(e->g_hin, in_host, bytes);
    CK(cudaGraphLaunch(e->g_exec, e->stream));
    e->launches += e->g_kernels;
    g_launches += e->g_kernels;
    CK(cudaStreamSynchronize(e->stream));
    memcpy(out_host, e->g_hout, obytes);
    *done = true;
    return 0;
}
}  // namespace

namespace {
// Host-buffer block steps: block b of this engine's channels starts at in_host + b*stride (stride == n_channels*B for a
// dense array; larger when the engine owns a channel range of a wider array) and out_host + b*out_stride (the output count
// of a matrix engine differs from its input count).  wait == false returns once everything
// is enqueued (engine_process_wait completes it) so that one host thread can keep several devices busy.
int engine_process_wait(irb_engine* e) {
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->s_out));
    CK(cudaStreamSynchronize(e->stream));
    e->pipe_pending = false;
    return 0;
}

int engine_process_enqueue(irb_engine* e, const void* in_host, int in_fmt, void* out_host, int out_fmt, int n_blocks, size_t stride, size_t out_stride, bool allow_graph) {
    CK(cudaSetDevice(e->device));
    int rc = engine_check_binding(e);
    if (rc) return rc;
    const size_t blk = e->in_blk(), oblk = e->out_blk();              // elements; strides too
    const size_t isz = fmt_size(in_fmt), osz = fmt_size(out_fmt);
    if (n_blocks == 1) {
        if (e->pipe_pending && (rc = engine_process_wait(e))) return rc;               // submitted blocks still own the staging slots
        // a live callback: one block in, one block out.  Small blocks replay a captured graph (one launch); larger ones
        // run copy, kernels, copy back to back on the engine's stream -- no cross-stream events to wait on.
        if (allow_graph) {
            bool done = false;
            if ((rc = engine_process_one_graphed(e, in_host, in_fmt, out_host, out_fmt, &done)) || done) return rc;
        }
        const int rows = tile_rows(e->M);
        const int tiles = (e->active + rows - 1) / rows;
        // (a matrix engine always takes the one-range form: its launch covers every group)
        const int groups = (e->timing || e->matrix() || isz * blk < (4u << 20)) ? 1 : (int) std::min<long long>(kMaxGroups, tiles / (4LL * e->num_sms) > 0 ? tiles / (4LL * e->num_sms) : 1);
        if (groups <= 1) {
            CK(cudaMemcpyAsync(e->io_in[0].p, in_host, isz * blk, cudaMemcpyHostToDevice, e->stream));
            if ((rc = engine_step_device(e, e->io_in[0].p, in_fmt, e->io_out[0].p, out_fmt))) return rc;
            CK(cudaMemcpyAsync(out_host, e->io_out[0].p, osz * oblk, cudaMemcpyDeviceToHost, e->stream));
            return 0;
        }
        // A large block: cut the channels into groups of whole tiles and pipeline upload | kernels | download across the
        // groups, so the block's latency is about its kernel time plus ONE group's copies instead of kernel time plus
        // all copies (what keeps a live feed of tens of thousands of channels inside its block period).
        if (e->ev_grp.empty()) {
            e->ev_grp.resize(2 * kMaxGroups, nullptr);
            for (auto& ev : e->ev_grp) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        }
        for (int g = 0; g < groups; ++g) {
            const int c0 = (int) ((long long) tiles * g / groups) * rows, c1 = std::min(e->active, (int) ((long long) tiles * (g + 1) / groups) * rows);
            const size_t off = (size_t) c0 * e->B, cnt = (size_t) (c1 - c0) * e->B;
            CK(cudaMemcpyAsync(fmt_at(e->io_in[0].p, in_fmt, off), fmt_at(in_host, in_fmt, off), isz * cnt, cudaMemcpyHostToDevice, e->s_in));
            CK(cudaEventRecord(e->ev_grp[2 * g], e->s_in));
            CK(cudaStreamWaitEvent(e->stream, e->ev_grp[2 * g], 0));
            if ((rc = engine_step_range(e, e->io_in[0].p, in_fmt, e->io_out[0].p, out_fmt, c0, c1 - c0, g == 0))) return rc;
            CK(cudaEventRecord(e->ev_grp[2 * g + 1], e->stream));
            CK(cudaStreamWaitEvent(e->s_out, e->ev_grp[2 * g + 1], 0));
            CK(cudaMemcpyAsync(fmt_at(out_host, out_fmt, off), fmt_at(e->io_out[0].p, out_fmt, off), osz * cnt, cudaMemcpyDeviceToHost, e->s_out));
        }
        return 0;
    }
    // three-stage pipeline over double-buffered device staging: upload b+1 | compute b | download b-1.  The staging slots
    // and their events persist across calls (pipe_seq), so back-to-back irb_engine_submit calls keep the pipeline full.
    for (int b = 0; b < n_blocks; ++b) {
        const int q = (int) (e->pipe_seq & 1);
        const bool reused = e->pipe_seq >= 2;
        ++e->pipe_seq;
        if (reused) CK(cudaStreamWaitEvent(e->s_in, e->ev_done[q], 0));            // the step two blocks back has consumed io_in[q]
        CK(cudaMemcpyAsync(e->io_in[q].p, fmt_at(in_host, in_fmt, b * stride), isz * blk, cudaMemcpyHostToDevice, e->s_in));
        CK(cudaEventRecord(e->ev_in[q], e->s_in));
        CK(cudaStreamWaitEvent(e->stream, e->ev_in[q], 0));
        if (reused) CK(cudaStreamWaitEvent(e->stream, e->ev_out[q], 0));           // its download has drained io_out[q]
        if ((rc = engine_step_device(e, e->io_in[q].p, in_fmt, e->io_out[q].p, out_fmt))) return rc;
        CK(cudaEventRecord(e->ev_done[q], e->stream));
        CK(cudaStreamWaitEvent(e->s_out, e->ev_done[q], 0));
        CK(cudaMemcpyAsync(fmt_at(out_host, out_fmt, b * out_stride), e->io_out[q].p, osz * oblk, cudaMemcpyDeviceToHost, e->s_out));
        CK(cudaEventRecord(e->ev_out[q], e->s_out));
    }
    e->pipe_pending = true;
    return 0;
}
}  // namespace

}  // extern "C"

// ---- IR loads: irb_engine_set_irs / _stage_irs and the group forms, one k_ir_load launch per chunk (irb_ir_load.cuh) ----------
namespace {
constexpr size_t kLoadSlotBytes = 64ull << 20;        // host sources: taps staged per chunk and side; two chunks in flight

// the partition count set_ir has always used: float ceil (fp/convolution.cpp:52)
int parts_for(int n_taps, int B) { return (int) std::ceil((float) n_taps / (float) B); }

// One load into one engine: row j (local IR ids[j]) is row rows[j] of the caller's array taps / right with stride ld.
struct LoadSpec {
    std::vector<int> ids, rows;
    const float* taps = nullptr;
    const float* right = nullptr;
    long long ld = 0;
    const int* n_taps = nullptr;       // [caller rows]; null: ld taps each
    int src_rows = 0;                  // rows of the caller's array: the last one may end at its own n_taps (no read past it)
    bool stage = false;
    int n_partitions = 0;
    int taps_of(int j) const { return n_taps ? n_taps[rows[j]] : (int) ld; }
};

// stage_ir's partition rule for a row
int stage_parts(const irb_engine* e, int ir, int nt, int n_partitions) {
    return n_partitions > 0 ? n_partitions : (e->h_nparts[ir] > 0 ? e->h_nparts[ir] : parts_for(nt, e->B));
}

// the argument errors a load's rows carry whatever the engine: null ids or taps, n < 1, a row without taps or longer than ld,
// a repeated id.  Checked before the engine itself, so that they are reported without a device.
int rows_check(int n, const int* ids, const float* taps, long long ld, const int* n_taps) {
    if (!ids || !taps) return fail(IRB_ERR_ARG, "ir_ids or taps null");
    if (n < 1) return fail(IRB_ERR_ARG, "n %d < 1", n);
    if (!n_taps && ld > 0x7fffffffLL) return fail(IRB_ERR_ARG, "ld %lld: rows of more than 2^31 - 1 taps", ld);
    for (int j = 0; j < n; ++j) {
        const long long nt = n_taps ? n_taps[j] : ld;
        if (nt < 1) return fail(IRB_ERR_ARG, "n_taps[%d] = %lld < 1", j, nt);
        if (ld < nt) return fail(IRB_ERR_ARG, "ld %lld < n_taps[%d] = %lld", ld, j, nt);
    }
    std::vector<std::pair<int, int>> v((size_t) n);
    for (int j = 0; j < n; ++j) v[j] = {ids[j], j};
    std::sort(v.begin(), v.end());
    for (int j = 1; j < n; ++j)
        if (v[j].first == v[j - 1].first) return fail(IRB_ERR_ARG, "ir_ids[%d] = %d repeats ir_ids[%d]", v[j].second, v[j].first, v[j - 1].second);
    return 0;
}

// the argument errors that depend on the engine (rows_check passed): an id outside [0, n_irs), more taps or partitions than the ring
int load_check(const irb_engine* e, const LoadSpec& s) {
    for (size_t j = 0; j < s.ids.size(); ++j) {
        const int ir = s.ids[j], nt = s.taps_of((int) j);
        if (ir < 0 || ir >= e->n_irs) return fail(IRB_ERR_ARG, "ir_ids[%d] = %d outside [0, %d)", s.rows[j], ir, e->n_irs);
        if (!s.stage && (long long) nt > (long long) e->B * e->ring)
            return fail(IRB_ERR_ARG, "n_taps[%d] = %d outside [1, %lld]", s.rows[j], nt, (long long) e->B * e->ring);
        if (s.stage) {
            const int P = stage_parts(e, ir, nt, s.n_partitions);
            if (P > e->ring) return fail(IRB_ERR_ARG, "row %d: %d partitions exceed max_partitions %d", s.rows[j], P, e->ring);
        }
    }
    return 0;
}

// where the taps are: 1 device memory the engine's kernels read in place (its own device, or managed), 0 host memory
// (pageable or pinned), -1 device memory of another device
int taps_location(const void* p, int dev) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (at.type == cudaMemoryTypeManaged) return 1;
    if (at.type == cudaMemoryTypeDevice) return at.device == dev ? 1 : -1;
    return 0;
}
int sources_location(const float* taps, const float* right, int dev, int* loc) {
    const int a = taps_location(taps, dev), b = right ? taps_location(right, dev) : a;
    if (a < 0 || b < 0) return fail(IRB_ERR_ARG, "taps in device memory of another device than the engine's %d", dev);
    if (a != b) return fail(IRB_ERR_ARG, "taps and right must both be host memory or both device memory");
    *loc = a;
    return 0;
}

template <int M>
int launch_ir_load_t(const irb::IrLoadArgs& a, long long grid, cudaStream_t st) {
    irb::k_ir_load<M><<<(unsigned) grid, irb::kThreads, 0, st>>>(a);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
int launch_ir_load(int M, const irb::IrLoadArgs& a, long long grid, cudaStream_t st) { IRB_DISPATCH_M(M, launch_ir_load_t<MM>(a, grid, st)); }

// Enqueue a checked load on the engine's stream; engine_load_wait completes it.  Everything that can fail for want of memory (new
// round-robin buffers, a larger item table, pooled staging, events) is acquired first, into locals: a failure there returns
// with the engine exactly as it was.  Only then does the host state change (partition counts, round-robin buffers and list, with
// set_ir's / stage_ir's per-IR rules), the device tables rr_ptrs, rr_list and nparts follow, and after them the copies and kernels.
// Host taps go through staging in chunks of whole rows: the upload of chunk k+1 (copy stream s_in) overlaps the transform of chunk
// k (the engine's stream).  Device taps are read in place by one launch.
int engine_load_enqueue(irb_engine* e, const LoadSpec& s, bool on_dev) {
    CK(cudaSetDevice(e->device));
    if (e->pipe_pending) { int rc = engine_process_wait(e); if (rc) return rc; }      // s_in and the stream are free
    const int n = (int) s.ids.size(), B = e->B;
    const long long cap = (long long) B * e->ring;
    // ---- plan, from the state as it is: per row the samples read, partitions, a spectra row, a cleared ring (first staging),
    // a round-robin buffer row, an rr_pos restart
    std::vector<int> len(n), P(n);
    std::vector<char> xf(n), clr(n), rr(n), restart(n), fresh(n);
    int lo = e->n_irs, hi = -1, n_fresh = 0;
    for (int j = 0; j < n; ++j) {
        const int ir = s.ids[j], nt = s.taps_of(j);
        lo = std::min(lo, ir); hi = std::max(hi, ir);
        if (!s.stage) {
            P[j] = parts_for(nt, B); len[j] = nt; xf[j] = 1; rr[j] = e->rr_buf[ir] != nullptr;
        } else {
            P[j] = stage_parts(e, ir, nt, s.n_partitions);
            len[j] = (int) std::min<long long>(nt, (long long) P[j] * B);      // taps beyond the partitions are never read
            rr[j] = 1;
            clr[j] = P[j] != e->h_nparts[ir] && e->h_nparts[ir] == 0;         // nothing was ever loaded: partitions fade in from cleared spectra
            fresh[j] = !e->rr_buf[ir];
            n_fresh += fresh[j];
        }
        restart[j] = rr[j] && P[j] != e->h_nparts[ir];
    }
    // chunks of whole rows [j0, j1), row k of a chunk staged at k * w (w: the longest row of the chunk); device taps: one chunk
    struct Chunk { int j0, j1, w; size_t tab, n_x, n_s; long long grid; };
    std::vector<Chunk> chunks;
    const size_t slot = on_dev ? 0 : std::max(kLoadSlotBytes / sizeof(float), (size_t) *std::max_element(len.begin(), len.end()));
    for (int j = 0; j < n;) {
        Chunk c{j, j, 0, 0, 0, 0, 0};
        while (c.j1 < n && (on_dev || (size_t) (c.j1 - c.j0 + 1) * (size_t) std::max(c.w, len[c.j1]) <= slot)) c.w = std::max(c.w, len[c.j1++]);
        chunks.push_back(c);
        j = c.j1;
    }
    std::vector<irb::IrLoadItem> tab;
    const long long rows_per_tile = tile_rows(e->M), pieces = (cap + irb::kPiece - 1) / irb::kPiece;
    for (auto& c : chunks) {
        c.tab = tab.size();
        auto off = [&](int j) { return on_dev ? (long long) s.rows[j] * s.ld : (long long) (j - c.j0) * c.w; };
        for (int j = c.j0; j < c.j1; ++j)
            if (xf[j] || clr[j]) tab.push_back({off(j), len[j], s.ids[j], xf[j] ? P[j] : 0, 0});
        c.n_x = tab.size() - c.tab;
        for (int j = c.j0; j < c.j1; ++j)
            if (rr[j]) tab.push_back({off(j), len[j], s.ids[j], restart[j] ? 1 : 0, 0});
        c.n_s = tab.size() - c.tab - c.n_x;
        c.grid = ((long long) c.n_x * e->ring + rows_per_tile - 1) / rows_per_tile + (long long) c.n_s * pieces;
        if (c.grid > 0x7fffffffLL) return fail(IRB_ERR_ARG, "a load of %lld tiles exceeds one launch", c.grid);
    }
    // a row stride above the copy engine's largest pitch: one copy per row instead of 2-D copies
    int max_pitch = 0;
    CK(cudaDeviceGetAttribute(&max_pitch, cudaDevAttrMaxPitch, e->device));
    const bool pitched = (long long) sizeof(float) * s.ld <= (long long) max_pitch;
    // ---- acquire: every allocation of the load, into locals
    std::vector<std::unique_ptr<DevBuf>> bufs((size_t) n);
    for (int j = 0; j < n; ++j) {
        if (!fresh[j]) continue;
        bufs[j].reset(new (std::nothrow) DevBuf);
        if (!bufs[j]) return fail(IRB_ERR_ARG, "out of host memory");
        if (int rc = bufs[j]->alloc(sizeof(float) * (size_t) cap, false)) { cudaGetLastError(); return rc; }      // an OOM is not left pending
    }
    DevBuf new_tab;
    size_t new_tab_cap = 0;
    if (tab.size() > e->ld_tab_cap) {
        new_tab_cap = std::max<size_t>(tab.size(), 1024);
        if (int rc = new_tab.alloc(sizeof(irb::IrLoadItem) * new_tab_cap, false)) { cudaGetLastError(); return rc; }
    }
    const int sides = s.right ? 2 : 1;
    const bool multi = chunks.size() > 1;
    std::unique_ptr<irbh::ScratchBuf> staging;
    float* stage_base = nullptr;
    size_t side_stride = 0, slot_stride = 0;             // floats between the sides of a slot, between the slots
    if (!on_dev) {                                       // the engine's own buffer when one chunk fits it, else two slots per side from the pool
        const size_t need = multi ? slot : (size_t) (chunks[0].j1 - chunks[0].j0) * chunks[0].w;
        if (!multi && need <= (size_t) cap) {
            stage_base = e->taps.as<float>(); side_stride = (size_t) cap;
        } else {
            staging.reset(new (std::nothrow) irbh::ScratchBuf);
            if (!staging) return fail(IRB_ERR_ARG, "out of host memory");
            if (int rc = staging->alloc(sizeof(float) * need * sides * (multi ? 2 : 1), false)) { cudaGetLastError(); return rc; }
            stage_base = staging->as<float>(); side_stride = need; slot_stride = need * sides;
        }
        if (multi && !e->ld_ev[3]) {
            cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
            for (auto& x : ev)
                if (cudaEventCreateWithFlags(&x, cudaEventDisableTiming) != cudaSuccess) {
                    for (auto y : ev) if (y) cudaEventDestroy(y);
                    return fail(IRB_ERR_CUDA, "event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
                }
            std::copy(ev, ev + 4, e->ld_ev);
        }
    }
    if (new_tab_cap) {                                   // the old table's last reader finished with the previous load's wait
        std::swap(e->ld_tab.p, new_tab.p);
        e->ld_tab_cap = new_tab_cap;
    }
    // ---- commit the host state; nothing below allocates
    std::vector<int> list = e->h_rr_list;
    for (int j = 0; j < n; ++j) if (fresh[j]) list.push_back(s.ids[j]);
    if (n_fresh) {
        std::vector<const float*> ptrs((size_t) e->n_irs, nullptr);
        for (int ir = 0; ir < e->n_irs; ++ir) if (e->rr_buf[ir]) ptrs[ir] = e->rr_buf[ir]->as<float>();
        for (int j = 0; j < n; ++j) if (fresh[j]) ptrs[s.ids[j]] = bufs[j]->as<float>();
        CK(cudaMemcpyAsync(e->rr_ptrs.p, ptrs.data(), sizeof(float*) * ptrs.size(), cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->rr_list.p, list.data(), sizeof(int) * list.size(), cudaMemcpyHostToDevice, e->stream));
    }
    for (int j = 0; j < n; ++j) {
        const int ir = s.ids[j];
        if (fresh[j]) { e->rr_buf[ir] = std::move(bufs[j]); e->bytes += sizeof(float) * (size_t) cap; }
        if (P[j] != e->h_nparts[ir]) e->plan_dirty = true;
        e->h_nparts[ir] = P[j];
    }
    e->h_rr_list.swap(list);
    e->ld_stage = std::move(staging);                    // held until engine_load_wait: copies and kernels read it
    CK(cudaMemcpyAsync(e->nparts.as<int>() + lo, e->h_nparts.data() + lo, sizeof(int) * (size_t) (hi - lo + 1), cudaMemcpyHostToDevice, e->stream));
    if (!tab.empty()) CK(cudaMemcpyAsync(e->ld_tab.p, tab.data(), sizeof(irb::IrLoadItem) * tab.size(), cudaMemcpyHostToDevice, e->stream));
    // ---- copies and kernels
    const cudaStream_t cs = multi ? e->s_in : e->stream;
    for (size_t ci = 0; ci < chunks.size(); ++ci) {
        const Chunk& c = chunks[ci];
        const int q = (int) (ci & 1);
        irb::IrLoadArgs a{};
        a.items = e->ld_tab.as<irb::IrLoadItem>() + c.tab; a.n_x = (int) c.n_x; a.n_s = (int) c.n_s;
        a.B = B; a.ring = e->ring; a.H = e->H.as<float2>(); a.ir_stride = (long long) e->ring * e->M;
        a.h_reps = e->h_reps; a.h_rep_stride = e->h_rep_stride(); a.W = e->W;
        a.rr_taps = e->rr_ptrs.as<float* const>(); a.rr_pos = e->rr_pos.as<int>();
        if (on_dev) {
            a.src = s.taps; a.src2 = s.right;
        } else {
            float* dst = stage_base + q * slot_stride;
            if (multi && ci >= 2) CK(cudaStreamWaitEvent(cs, e->ld_ev[2 + q], 0));      // the transform two chunks back has read this slot
            for (int side = 0; side < sides; ++side) {
                const float* src = side ? s.right : s.taps;
                float* d = dst + side * side_stride;
                // runs of consecutive caller rows, one 2-D copy each; the caller's last row alone, at its own length
                for (int j = c.j0; j < c.j1;) {
                    int k = j + 1;
                    while (pitched && k < c.j1 && s.rows[k] == s.rows[k - 1] + 1 && s.rows[k] != s.src_rows - 1) ++k;
                    if (k == j + 1) CK(cudaMemcpyAsync(d + (size_t) (j - c.j0) * c.w, src + (long long) s.rows[j] * s.ld, sizeof(float) * len[j], cudaMemcpyHostToDevice, cs));
                    else CK(cudaMemcpy2DAsync(d + (size_t) (j - c.j0) * c.w, sizeof(float) * c.w, src + (long long) s.rows[j] * s.ld, sizeof(float) * s.ld,
                                              sizeof(float) * c.w, k - j, cudaMemcpyHostToDevice, cs));
                    j = k;
                }
            }
            if (multi) {
                CK(cudaEventRecord(e->ld_ev[q], cs));
                CK(cudaStreamWaitEvent(e->stream, e->ld_ev[q], 0));
            }
            a.src = dst; a.src2 = s.right ? dst + side_stride : nullptr;
        }
        if (c.grid > 0) {
            if (int rc = launch_ir_load(e->M, a, c.grid, e->stream)) return rc;
            e->launches += 1;
        }
        if (multi) CK(cudaEventRecord(e->ld_ev[2 + q], e->stream));
    }
    return 0;
}
// the load's work is in place: both streams drained (an early error can leave copies running on s_in), then the pooled staging
// goes back to the pool
int engine_load_wait(irb_engine* e) {
    CK(cudaSetDevice(e->device));
    const cudaError_t ci = cudaStreamSynchronize(e->s_in);
    const cudaError_t ce = cudaStreamSynchronize(e->stream);
    e->ld_stage.reset();
    CK(ci);
    CK(ce);
    return 0;
}

int engine_load(irb_engine* e, int n, const int* ids, const float* taps, const float* right, long long ld, const int* n_taps, bool stage, int n_partitions) {
    int rc = rows_check(n, ids, taps, ld, n_taps);
    if (rc) return rc;
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    LoadSpec s;
    s.ids.assign(ids, ids + n);
    s.rows.resize(n);
    for (int j = 0; j < n; ++j) s.rows[j] = j;
    s.taps = taps; s.right = right; s.ld = ld; s.n_taps = n_taps; s.src_rows = n; s.stage = stage; s.n_partitions = n_partitions;
    if ((rc = load_check(e, s))) return rc;
    int loc = 0;
    if ((rc = sources_location(taps, right, e->device, &loc))) return rc;
    rc = engine_load_enqueue(e, s, loc == 1);
    const int w = engine_load_wait(e);
    return rc ? rc : w;
}
}  // namespace

extern "C" {
int irb_engine_set_irs(irb_engine* e, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps) {
    return engine_load(e, n, ir_ids, taps, right, ld, n_taps, false, 0);
}
int irb_engine_stage_irs(irb_engine* e, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps, int n_partitions) {
    return engine_load(e, n, ir_ids, taps, right, ld, n_taps, true, n_partitions);
}

// Streams come and go: only channels [0, n_active) take part in the following block steps (their FDL rings advance, the
// others keep their state untouched); in/out arrays of the process calls are then [n_blocks][n_active][block_size].
// n_active must be a whole number of kernel tiles (irb_engine_tile_channels()) or n_channels.
int irb_engine_set_active_channels(irb_engine* e, int n_active) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    if (e->matrix()) return fail(IRB_ERR_STATE, "an IR-matrix engine always runs all its groups");
    if (n_active < 1 || n_active > e->n_chans) return fail(IRB_ERR_ARG, "n_active %d outside [1, %d]", n_active, e->n_chans);
    if (n_active != e->n_chans && n_active % tile_rows(e->M)) return fail(IRB_ERR_ARG, "n_active %d is not a multiple of the %d channels of a kernel tile", n_active, tile_rows(e->M));
    if (e->pipe_pending) { int rc = engine_process_wait(e); if (rc) return rc; }
    e->active = n_active;
    e->plan_dirty = true;
    return 0;
}
int irb_engine_active_channels(const irb_engine* e) { return e ? e->active : fail(IRB_ERR_ARG, "engine is null"); }

int irb_engine_process(irb_engine* e, const float* in_host, float* out_host, int n_blocks) {
    return irb_engine_process_pcm(e, in_host, IRB_SAMPLE_F32, out_host, IRB_SAMPLE_F32, n_blocks);
}
int irb_engine_process_pcm(irb_engine* e, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks) {
    if (!fmt_valid(in_format) || !fmt_valid(out_format)) return fail(IRB_ERR_ARG, "sample format %d / %d is not an irb_sample_format", in_format, out_format);
    if (!e || !in_host || !out_host) return fail(IRB_ERR_ARG, "null argument");
    if (n_blocks < 0) return fail(IRB_ERR_ARG, "n_blocks < 0");
    int rc = engine_process_enqueue(e, in_host, in_format, out_host, out_format, n_blocks, e->in_blk(), e->out_blk(), true);
    if (rc) return rc;
    return engine_process_wait(e);
}

// Asynchronous host path for a continuous feed: submit returns once the copies and kernels of the blocks are enqueued
// (the host arrays must stay valid and pinned until the wait); consecutive submits keep the three-stage pipeline full
// instead of draining it at every call.  irb_engine_wait returns when everything submitted so far is back in host memory.
int irb_engine_submit(irb_engine* e, const float* in_host, float* out_host, int n_blocks) {
    return irb_engine_submit_pcm(e, in_host, IRB_SAMPLE_F32, out_host, IRB_SAMPLE_F32, n_blocks);
}
int irb_engine_submit_pcm(irb_engine* e, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks) {
    if (!fmt_valid(in_format) || !fmt_valid(out_format)) return fail(IRB_ERR_ARG, "sample format %d / %d is not an irb_sample_format", in_format, out_format);
    if (n_blocks == 1) return fail(IRB_ERR_ARG, "irb_engine_submit takes at least two blocks per call (one block at a time is irb_engine_process)");
    if (!e || !in_host || !out_host) return fail(IRB_ERR_ARG, "null argument");
    if (n_blocks < 0) return fail(IRB_ERR_ARG, "n_blocks < 0");
    if (n_blocks == 0) return 0;
    return engine_process_enqueue(e, in_host, in_format, out_host, out_format, n_blocks, e->in_blk(), e->out_blk(), false);
}
int irb_engine_wait(irb_engine* e) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    return engine_process_wait(e);
}

// The order of one plug-in callback (PluginProcessor.cpp:421-518): EVERY block completed by the callback is transformed
// into the FDL first (:421-445), then the blocks are convolved one after the other (:452-518), each preceded by one
// round-robin IR refresh (:455-461).  With n_blocks > 1 (host block > processBlockSize) the oldest partitions of the
// earlier blocks therefore meet slots already overwritten by the later blocks of the same callback whenever
// max_partitions < partitions + n_blocks - 1 -- the reference's behaviour, kept (create the engine with a larger ring
// to avoid it).  in/out: HOST [n_blocks][n_channels][block_size].
int irb_engine_process_callback(irb_engine* e, const float* in_host, float* out_host, int n_blocks) {
    if (!e || !in_host || !out_host) return fail(IRB_ERR_ARG, "null argument");
    if (n_blocks < 0) return fail(IRB_ERR_ARG, "n_blocks < 0");
    if (e->matrix()) return fail(IRB_ERR_STATE, "an IR-matrix engine has no callback-order path: use irb_engine_process");
    if (n_blocks > e->ring) return fail(IRB_ERR_ARG, "%d blocks in one callback exceed the FDL ring of %d slots", n_blocks, e->ring);
    if (n_blocks == 0) return 0;
    CK(cudaSetDevice(e->device));
    int rc = engine_check_binding(e);
    if (rc) return rc;
    const size_t blk = (size_t) e->B * e->active;
    if (e->cb_blocks < n_blocks) {
        e->cb_in.reset(new (std::nothrow) DevBuf); e->cb_out.reset(new (std::nothrow) DevBuf);
        if (!e->cb_in || !e->cb_out) return fail(IRB_ERR_ARG, "out of host memory");
        e->cb_blocks = 0;
        const size_t cap = sizeof(float) * (size_t) e->B * e->n_chans * n_blocks;       // sized for every channel: the active count may grow later
        if ((rc = e->cb_in->alloc(cap, false)) || (rc = e->cb_out->alloc(cap, false))) return rc;
        e->cb_blocks = n_blocks;
    }
    float* din = e->cb_in->as<float>();
    float* dout = e->cb_out->as<float>();
    CK(cudaMemcpyAsync(din, in_host, sizeof(float) * blk * n_blocks, cudaMemcpyHostToDevice, e->stream));
    for (int b = 0; b < n_blocks; ++b)
        if ((rc = engine_launch_fwd(e, din + b * blk, IRB_SAMPLE_F32, true, false, 0, e->active))) return rc;
    for (int b = 0; b < n_blocks; ++b) {
        if ((rc = engine_launch_fwd(e, nullptr, IRB_SAMPLE_F32, false, true, 0, e->active))) return rc;
        if ((rc = engine_launch_mac(e, dout + b * blk, IRB_SAMPLE_F32, n_blocks - 1 - b, nullptr, IRB_SAMPLE_F32, 0, e->active))) return rc;
    }
    CK(cudaMemcpyAsync(out_host, dout, sizeof(float) * blk * n_blocks, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

int irb_engine_set_timing(irb_engine* e, int enable) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    if (enable && e->tev.empty()) {
        e->tev.resize(3 * (size_t) kTimingCap, nullptr);
        e->tev_mid.assign((size_t) kTimingCap, 0);
        for (auto& ev : e->tev) CK(cudaEventCreate(&ev));
    }
    e->timing = enable != 0;
    e->t_rec = 0;
    return 0;
}

int irb_engine_get_timings(irb_engine* e, float* step_ms, float* mac_ms, int max_steps) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    const int n = e->t_rec < max_steps ? e->t_rec : max_steps;
    for (int i = 0; i < n; ++i) {
        if (step_ms) CK(cudaEventElapsedTime(step_ms + i, e->tev[3 * i], e->tev[3 * i + 2]));
        if (mac_ms) CK(cudaEventElapsedTime(mac_ms + i, e->tev[3 * i + (e->tev_mid[i] ? 1 : 0)], e->tev[3 * i + 2]));
    }
    return n;
}

int irb_engine_synchronize(irb_engine* e) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

size_t irb_engine_state_bytes(const irb_engine* e) { return e ? e->bytes : 0; }
int irb_engine_fft_size(const irb_engine* e) { return e ? 2 * e->M : fail(IRB_ERR_ARG, "engine is null"); }
int irb_engine_partitions(const irb_engine* e, int ir_id) {
    if (!e || ir_id < 0 || ir_id >= e->n_irs) return fail(IRB_ERR_ARG, "bad engine or ir_id");
    return e->h_nparts[ir_id];
}
long long irb_engine_launch_count(const irb_engine* e) { return e ? e->launches : 0; }

int irb_engine_read_ir_spectrum(irb_engine* e, int ir_id, int part, float* out_packed) {
    if (!e || !out_packed || ir_id < 0 || ir_id >= e->n_irs || part < 0 || part >= e->ring) return fail(IRB_ERR_ARG, "bad argument");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(out_packed, e->H.as<float2>() + ((size_t) ir_id * e->ring + part) * e->M, sizeof(float2) * e->M, cudaMemcpyDeviceToHost));
    return 0;
}
int irb_engine_read_fdl_spectrum(irb_engine* e, int chan, int age, float* out_packed) {
    if (!e || !out_packed || chan < 0 || chan >= e->n_chans || age < 0 || age >= e->ring) return fail(IRB_ERR_ARG, "bad argument");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    int head = 0;
    CK(cudaMemcpy(&head, e->head.as<int>() + chan, sizeof(int), cudaMemcpyDeviceToHost));
    const int slot = ((head - age) % e->ring + e->ring) % e->ring;
    const size_t off = (size_t) (chan / e->fdl_group) * e->fdl_group_stride() + ((size_t) slot * e->fdl_group + chan % e->fdl_group) * e->M;
    CK(cudaMemcpy(out_packed, e->fdl.as<float2>() + off, sizeof(float2) * e->M, cudaMemcpyDeviceToHost));
    return 0;
}

// fp::ir::IRtoRealFFTRaw (fp/ir.cpp:106-147): the IR cut into len/part_size + 1 partitions of part_size samples, each
// zero-padded to 2*part_size, transformed, stored as {Re X[0], Re X[N/2], re1, im1, ...} -- exactly the packed spectrum
// rows of the engine.  out: (len/part_size + 1) * 2*part_size floats.  part_size must be a power of two in [16, 2048].
int irb_ir_to_real_fft_raw(const float* x, int len, int part_size, float* out) {
    if (!x || !out || len < 1) return fail(IRB_ERR_ARG, "bad argument");
    if (part_size < 16 || part_size > kMaxM || (part_size & (part_size - 1))) return fail(IRB_ERR_ARG, "part_size %d must be a power of two in [16, %d]", part_size, kMaxM);
    const int M = part_size, parts = len / part_size + 1, dev = irbh::g_device;
    CK(cudaSetDevice(dev));
    const float2* W = nullptr;
    int rc = irbh::twiddles(dev, M, &W);
    if (rc) return rc;
    irbh::ScratchBuf dx, dH;
    irbh::StreamGuard sg;              // declared after the buffers: its destructor drains the stream before they go back to the pool
    if ((rc = sg.create())) return rc;
    if ((rc = dx.alloc(sizeof(float) * (size_t) len, false)) || (rc = dH.alloc(sizeof(float2) * (size_t) M * parts, true))) return rc;
    CK(cudaMemcpyAsync(dx.p, x, sizeof(float) * (size_t) len, cudaMemcpyHostToDevice, sg.s));
    irb::FwdArgs f{};
    f.src = dx.as<float>(); f.src_chan_stride = 0; f.L = len; f.B = part_size; f.blocks_per_chan = parts; f.n_rows = parts;
    f.dst = dH.as<float2>(); f.dst_chan_stride = 0; f.W = W;
    if ((rc = launch_fwd(M, f, sg.s))) return rc;
    CK(cudaMemcpyAsync(out, dH.p, sizeof(float2) * (size_t) M * parts, cudaMemcpyDeviceToHost, sg.s));
    CK(cudaStreamSynchronize(sg.s));
    return 0;
}

// fp::convolution::convolvePeriodic (fp/convolution.cpp:14-242) with every block processed at once:
// all audio blocks are transformed in one launch, output block k sums X[k-p]*H[p] over the partitions
// p <= k in ascending order (the reference's own order, :171-202), and the overlap of block k-1 is added
// afterwards (:210-213).  Feeding zero blocks after the input ends is the reference's tail loop
// (:150-153,166-167) because the partitions it skips there would only meet slots that hold zeros here.
int irb_convolve_periodic(const float* x, int ch_x, int len_x, const float* h, int ch_h, int len_h, int block_size, float* out) {
    if (!x || !h || !out) return fail(IRB_ERR_ARG, "null argument");
    if (len_x < 1 || len_h < 1 || ch_x < 1 || ch_h < 1) return fail(IRB_ERR_ARG, "empty input");
    const long long Lout = (long long) len_x + len_h - 1;
    memset(out, 0, sizeof(float) * (size_t) ch_x * Lout);
    if (!((ch_x == 1 || ch_x == 2) && (ch_h == 1 || ch_h == 2)))
        return fail(IRB_ERR_LAYOUT, "audio has %d channels and the IR %d: only mono/stereo layouts exist (fp/convolution.cpp:28-42)", ch_x, ch_h);
    if (block_size < 1) return fail(IRB_ERR_ARG, "block_size %d < 1", block_size);
    if (Lout > 0x7fffffffLL) return fail(IRB_ERR_ARG, "output too long");
    CK(cudaSetDevice(irbh::g_device));
    // What the reference's block size decides about the RESULT is only how much of the linear convolution gets written:
    // iters = Lx/B + P blocks, the last overlap never flushed (:104-233,233-238).  Every sample before that point is the
    // same linear convolution for any partitioning (SURVEY KA4), so block sizes above the block kernels' range are
    // computed with the largest supported block and cut at the reference's length.
    const int P_ref = (int) std::ceil((float) len_h / (float) block_size);
    const long long iters_ref = (long long) len_x / block_size + P_ref;
    const long long Lw = Lout < iters_ref * block_size ? Lout : iters_ref * block_size;
    const bool native = half_size_for_block(block_size) <= kMaxM;
    const int B = native ? block_size : kMaxM;
    const int M = half_size_for_block(B);
    const float2* W = nullptr;
    int rc = irbh::twiddles(irbh::g_device, M, &W);
    if (rc) return rc;
    const int P = (int) std::ceil((float) len_h / (float) B);
    const int iters = native ? (int) iters_ref : (int) ((Lw + B - 1) / B);      // blocks past the input are zero blocks
    const int rows = tile_rows(M);
    const int bpc = (iters + rows - 1) / rows * rows;      // padded so no tile straddles two channels
    const bool fold = (ch_h == 2 && ch_x == 1);            // IRStereoAudioMono: (L+R)/2, :120-121
    const int n_ir = (ch_h == 2 && ch_x == 2) ? 2 : 1;     // IRStereoAudioStereo is channel-wise, :176-181

    irbh::ScratchBuf dx, dh, dX, dH, dout, dtail, dnp, dir;
    irbh::StreamGuard sg;              // declared after the buffers: an early return drains the stream before they go back to the pool
    if ((rc = sg.create())) return rc;
    cudaStream_t st = sg.s;
    const size_t spec = sizeof(float2) * (size_t) M;
    if ((rc = dx.alloc(sizeof(float) * (size_t) ch_x * len_x, false)) || (rc = dh.alloc(sizeof(float) * (size_t) ch_h * len_h, false)) ||
        (rc = dX.alloc(spec * bpc * ch_x, false)) || (rc = dH.alloc(spec * P * n_ir, false)) ||
        (rc = dout.alloc(sizeof(float) * (size_t) ch_x * Lout, true)) || (rc = dtail.alloc(sizeof(float) * (size_t) B * bpc * ch_x, false)) ||
        (rc = dnp.alloc(sizeof(int) * 2, false)) || (rc = dir.alloc(sizeof(int) * 2, false)))
        return rc;
    CK(cudaMemcpyAsync(dx.p, x, sizeof(float) * (size_t) ch_x * len_x, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(dh.p, h, sizeof(float) * (size_t) ch_h * len_h, cudaMemcpyHostToDevice, st));
    const int np[2] = {P, P};
    const int irmap[2] = {0, n_ir == 2 ? 1 : 0};
    CK(cudaMemcpyAsync(dnp.p, np, sizeof(np), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(dir.p, irmap, sizeof(irmap), cudaMemcpyHostToDevice, st));

    irbh::ComputeTimer tm;
    if ((rc = tm.init(st)) || (rc = tm.begin())) return rc;
    irb::FwdArgs fh{};                                      // IR partitions
    fh.src = dh.as<float>(); fh.src2 = fold ? dh.as<float>() + len_h : nullptr; fh.src_chan_stride = len_h; fh.L = len_h; fh.B = B;
    fh.blocks_per_chan = P; fh.n_rows = P * n_ir; fh.dst = dH.as<float2>(); fh.dst_chan_stride = (long long) P * M; fh.W = W;
    if ((rc = launch_fwd(M, fh, st))) return rc;
    irb::FwdArgs fx{};                                      // audio blocks (blocks past the input are zero)
    fx.src = dx.as<float>(); fx.src_chan_stride = len_x; fx.L = len_x; fx.B = B;
    fx.blocks_per_chan = bpc; fx.n_rows = bpc * ch_x; fx.dst = dX.as<float2>(); fx.dst_chan_stride = (long long) bpc * M; fx.W = W;
    if ((rc = launch_fwd(M, fx, st))) return rc;
    irb::MacArgs m{};
    m.fdl = dX.as<float2>(); m.fdl_chan_stride = (long long) bpc * M; m.head = nullptr; m.ring = bpc; m.blocks_per_chan = bpc;
    m.n_rows = bpc * ch_x; m.H = dH.as<float2>(); m.ir_stride = (long long) P * M; m.ir_of_chan = dir.as<int>(); m.nparts = dnp.as<int>();
    m.W = W; m.B = B; m.out = dout.as<float>(); m.out_chan_stride = Lout; m.Lout = (int) Lw; m.ov = nullptr; m.tail = dtail.as<float>();
    m.split_in = 1;
    mac_policy(m);
    if ((rc = launch_mac(M, true, false, 1, 148, m, st))) return rc;
    {
        const long long n = (long long) bpc * B * ch_x;
        irb::k_ola_tail<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>(dout.as<float>(), Lout, (int) Lw, dtail.as<float>(), B, bpc, ch_x);
        g_launches++;
        CK(cudaGetLastError());
    }
    if ((rc = tm.end())) return rc;
    CK(cudaMemcpyAsync(out, dout.p, sizeof(float) * (size_t) ch_x * Lout, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return tm.collect();
}

// ---- several GPUs driven from one process (SURVEY 8e): streams sharded by contiguous, tile-aligned channel ranges, shared
// IR spectra replicated on every device, per-channel IRs (n_irs == 0) living with their channel; no device-to-device
// traffic -- every device reads its channel range of the caller's arrays and writes its range of the output.
struct irb_group {
    std::vector<irb_engine*> eng;
    std::vector<int> begin;            // eng[i] owns channels [begin[i], begin[i+1])
    int B = 0, n_chans = 0, n_irs = 0;
    bool private_irs = false;
    int owner(int chan) const { int i = 0; while (i + 1 < (int) eng.size() && chan >= begin[i + 1]) ++i; return i; }
};

int irb_group_create(irb_group** out, const int* devices, int n_devices, int block_size, int max_partitions, int n_channels, int n_irs) {
    if (!out) return fail(IRB_ERR_ARG, "out is null");
    *out = nullptr;
    if (!devices || n_devices < 1) return fail(IRB_ERR_ARG, "no devices");
    if (block_size < 1 || half_size_for_block(block_size) > kMaxM) return fail(IRB_ERR_ARG, "block_size %d outside [1, %d]", block_size, kMaxM);
    if (n_channels < n_devices || n_irs < 0) return fail(IRB_ERR_ARG, "need at least one channel per device and n_irs >= 0");
    std::unique_ptr<irb_group> g(new (std::nothrow) irb_group);
    if (!g) return fail(IRB_ERR_ARG, "out of host memory");
    g->B = block_size; g->n_chans = n_channels; g->n_irs = n_irs; g->private_irs = n_irs == 0;
    const int rows = tile_rows(half_size_for_block(block_size));
    const int tiles = (n_channels + rows - 1) / rows;
    if (tiles < n_devices) return fail(IRB_ERR_ARG, "%d channels are fewer than one kernel tile (%d channels) per device", n_channels, rows);
    for (int i = 0; i <= n_devices; ++i) g->begin.push_back(std::min(n_channels, (int) ((long long) tiles * i / n_devices) * rows));
    for (int i = 0; i < n_devices; ++i) {
        irb_engine* e = nullptr;
        const int local = g->begin[i + 1] - g->begin[i];
        int rc = irb_engine_create(&e, devices[i], block_size, max_partitions, local, g->private_irs ? local : n_irs);
        if (rc) { for (auto* p : g->eng) irb_engine_destroy(p); return rc; }
        g->eng.push_back(e);
        if (g->private_irs) for (int c = 0; c < local; ++c) e->h_ir_of_chan[c] = c;      // channel c convolves with its own IR
        e->binding_dirty = true;
    }
    *out = g.release();
    return 0;
}
int irb_group_destroy(irb_group* g) {
    if (!g) return 0;
    for (auto* e : g->eng) irb_engine_destroy(e);
    delete g;
    return 0;
}
int irb_group_device_count(const irb_group* g) { return g ? (int) g->eng.size() : fail(IRB_ERR_ARG, "group is null"); }
int irb_group_channel_range(const irb_group* g, int index, int* begin, int* end) {
    if (!g || index < 0 || index >= (int) g->eng.size()) return fail(IRB_ERR_ARG, "bad group or index");
    if (begin) *begin = g->begin[index];
    if (end) *end = g->begin[index + 1];
    return 0;
}
// shared IRs (n_irs > 0): ir_id on every device.  Private IRs (n_irs == 0): ir_id is the CHANNEL whose IR this is.
int irb_group_set_ir(irb_group* g, int ir_id, const float* left, const float* right, int n_taps) {
    return irb_group_set_irs(g, 1, &ir_id, left, right, n_taps, &n_taps);
}
int irb_group_stage_ir(irb_group* g, int ir_id, const float* left, const float* right, int n_taps, int n_partitions) {
    return irb_group_stage_irs(g, 1, &ir_id, left, right, n_taps, &n_taps, n_partitions);
}
}  // extern "C"
namespace {
// rows of a private-IR group go to the device owning channel ir_ids[j] (as its local IR), rows of a shared-IR group to every
// device; all checks first, then every device's copies and kernels, then the waits
int group_load(irb_group* g, int n, const int* ids, const float* taps, const float* right, long long ld, const int* n_taps, bool stage, int n_partitions) {
    int rc = rows_check(n, ids, taps, ld, n_taps);
    if (rc) return rc;
    if (!g) return fail(IRB_ERR_ARG, "group is null");
    std::vector<LoadSpec> s(g->eng.size());
    for (auto& x : s) { x.taps = taps; x.right = right; x.ld = ld; x.n_taps = n_taps; x.src_rows = n; x.stage = stage; x.n_partitions = n_partitions; }
    for (int j = 0; j < n; ++j) {
        if (g->private_irs) {
            if (ids[j] < 0 || ids[j] >= g->n_chans) return fail(IRB_ERR_ARG, "ir_ids[%d]: channel %d outside [0, %d)", j, ids[j], g->n_chans);
            const int i = g->owner(ids[j]);
            s[i].ids.push_back(ids[j] - g->begin[i]); s[i].rows.push_back(j);
        } else {
            for (auto& x : s) { x.ids.push_back(ids[j]); x.rows.push_back(j); }
        }
    }
    for (size_t i = 0; i < s.size(); ++i) if ((rc = s[i].ids.empty() ? 0 : load_check(g->eng[i], s[i]))) return rc;
    int loc = 0;
    if ((rc = sources_location(taps, right, g->eng[0]->device, &loc))) return rc;
    if (loc != 0) return fail(IRB_ERR_ARG, "irb_group_* loads take host memory: the taps are device memory");
    size_t started = 0;
    for (; started < s.size() && !rc; ++started) rc = s[started].ids.empty() ? 0 : engine_load_enqueue(g->eng[started], s[started], false);
    for (size_t i = 0; i < started; ++i) { const int w = s[i].ids.empty() ? 0 : engine_load_wait(g->eng[i]); if (!rc) rc = w; }
    return rc;
}
}  // namespace
extern "C" {
int irb_group_set_irs(irb_group* g, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps) {
    return group_load(g, n, ir_ids, taps, right, ld, n_taps, false, 0);
}
int irb_group_stage_irs(irb_group* g, int n, const int* ir_ids, const float* taps, const float* right, long long ld, const int* n_taps, int n_partitions) {
    return group_load(g, n, ir_ids, taps, right, ld, n_taps, true, n_partitions);
}
int irb_group_bind(irb_group* g, int chan_begin, int chan_end, int ir_id) {
    if (!g) return fail(IRB_ERR_ARG, "group is null");
    if (g->private_irs) return fail(IRB_ERR_STATE, "a group created with n_irs == 0 binds every channel to its own IR");
    if (chan_begin < 0 || chan_end > g->n_chans || chan_begin > chan_end) return fail(IRB_ERR_ARG, "channel range [%d, %d) outside [0, %d)", chan_begin, chan_end, g->n_chans);
    for (size_t i = 0; i < g->eng.size(); ++i) {
        const int b = std::max(chan_begin, g->begin[i]), e = std::min(chan_end, g->begin[i + 1]);
        if (b < e) { int rc = irb_engine_bind(g->eng[i], b - g->begin[i], e - g->begin[i], ir_id); if (rc) return rc; }
    }
    return 0;
}
int irb_group_reset(irb_group* g) {
    if (!g) return fail(IRB_ERR_ARG, "group is null");
    for (auto* e : g->eng) { int rc = irb_engine_reset(e); if (rc) return rc; }
    return 0;
}
// in/out: HOST [n_blocks][n_channels][block_size] for ALL channels; every device is fed from one thread (enqueue all, then wait all)
int irb_group_process(irb_group* g, const float* in_host, float* out_host, int n_blocks) {
    return irb_group_process_pcm(g, in_host, IRB_SAMPLE_F32, out_host, IRB_SAMPLE_F32, n_blocks);
}
int irb_group_process_pcm(irb_group* g, const void* in_host, int in_format, void* out_host, int out_format, int n_blocks) {
    if (!fmt_valid(in_format) || !fmt_valid(out_format)) return fail(IRB_ERR_ARG, "sample format %d / %d is not an irb_sample_format", in_format, out_format);
    if (!g || !in_host || !out_host) return fail(IRB_ERR_ARG, "null argument");
    if (n_blocks < 0) return fail(IRB_ERR_ARG, "n_blocks < 0");
    const size_t stride = (size_t) g->B * g->n_chans;            // elements
    int rc = 0;
    size_t started = 0;
    for (; started < g->eng.size() && !rc; ++started) {
        const size_t off = (size_t) g->begin[started] * g->B;
        rc = engine_process_enqueue(g->eng[started], fmt_at(in_host, in_format, off), in_format, fmt_at(out_host, out_format, off), out_format, n_blocks, stride, stride, false);
    }
    for (size_t i = 0; i < started; ++i) { const int w = engine_process_wait(g->eng[i]); if (!rc) rc = w; }
    return rc;
}
size_t irb_group_state_bytes(const irb_group* g) {
    size_t n = 0;
    if (g) for (auto* e : g->eng) n += e->bytes;
    return n;
}

}  // extern "C"

// ---- internals reached by the bench-only translation unit (irb_benchaids.cu, include/irb_b200_bench.h) -------------------
namespace irbh {
int engine_set_stamps(irb_engine* e, unsigned long long* dev) {
    if (!e) return fail(IRB_ERR_ARG, "engine is null");
    e->stamps = dev;
    e->g_sig.n_rr = -1;                // a captured graph baked the old pointer in: re-capture
    return 0;
}
int engine_ir_copies(const irb_engine* e) { return e ? e->h_reps : fail(IRB_ERR_ARG, "engine is null"); }
// the pure FDL multiply-accumulate (no forward / inverse FFT) on the current state into n_channels * M complex
int engine_mac_only(irb_engine* e, float* acc_dev) {
    if (!e || !acc_dev) return fail(IRB_ERR_ARG, "null argument");
    CK(cudaSetDevice(e->device));
    int rc = engine_check_binding(e);
    if (rc) return rc;
    irb::MacArgs m{};
    fill_mac_args(e, m, 0, e->active);
    m.Y = (float2*) acc_dev;
    m.work = nullptr;
    rc = launch_mac(e->M, false, use_slots(e), e->cluster_dim, e->num_sms, m, e->stream);
    if (rc) return rc;
    e->launches += 1;
    return 0;
}
}  // namespace irbh
